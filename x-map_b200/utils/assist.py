"""Pipeline glue with the reference's names and signatures (xmap/utils/assist.py:9-215).

`sc` / `sqlContext` may be None (no Spark on the GPU boxes): results then come back as
rdd.LocalRDD objects; with a real SparkContext the flat AlterEgo records are parallelised
so downstream Spark code (MLlib ALS, the item-kNN stages) runs unchanged."""
from os import makedirs
from os.path import join
import time

from ..rdd import LocalRDD, context_of, records_of


def baseliner_clean_data_pipeline(sc, clean_tool, path_rawdata, is_debug, num_partition):
    """assist.py:9-21."""
    ctx = context_of(sc)
    parsed = clean_tool.parse_data(ctx.textFile(path_rawdata, 30))
    cleaned = clean_tool.clean_data(clean_tool.filter_data(parsed))
    if is_debug:
        return ctx.parallelize(clean_tool.take_partial_data(cleaned), num_partition)
    return cleaned if sc is None else ctx.parallelize(cleaned.collect(), num_partition)


def baseliner_split_data_pipeline(sc, split_tool, sourceRDD, targetRDD):
    """assist.py:24-39."""
    ctx = context_of(sc)
    overlap = ctx.broadcast(split_tool.find_overlap_user(sourceRDD, targetRDD).collect())
    ov_s, non_s = split_tool.distinguish_data(overlap, sourceRDD)
    ov_t, non_t = split_tool.distinguish_data(overlap, targetRDD)
    train, test = split_tool.split_data(non_s, ov_s, non_t, ov_t)
    if sc is None:
        return train, test
    return ctx.parallelize(train.collect()), ctx.parallelize(test.collect())


def baseliner_calculate_sim_pipeline(sc, itemsim_tool, trainRDD):
    """assist.py:66-77.  Builds the ratings layout + statistics on the GPU now; the returned RDD
    is lazy (its records materialise only if collected) and carries the device state that
    extender_pipeline consumes."""
    return itemsim_tool.calculate_item2item_sim(trainRDD)


def extender_pipeline(sc, sqlContext, itemsim_tool, extendsim_tool, item2item_simRDD):
    """assist.py:80-102: BB set, per-class top-k, X-SIM extension, all on the device."""
    from ..core.extender import _sim_handle
    return extendsim_tool.extend(_sim_handle(item2item_simRDD))


def extract_siminfo(sc, classfied_items):
    """assist.py:105-133 (host dictionaries; only for callers that want them)."""
    ctx = context_of(sc)
    recs = records_of(classfied_items)
    BB_info = LocalRDD((i, b) for i, b, n in recs if b is not None)
    NB_info = LocalRDD((i, n) for i, b, n in recs if n is not None)
    knn_BB = {i: dict((l[0], l[1:]) for l in b[0] + b[1]) for i, b in BB_info.collect()}
    knn_NB = {i: dict((l[0], l[1:]) for l in n[0] + n[1]) for i, n in NB_info.collect()}
    return BB_info, NB_info, ctx.broadcast(knn_BB), ctx.broadcast(knn_NB)


def generator_pipeline(privatemap_tool, trainRDD, extended_simRDD, private):
    """assist.py:136-150."""
    from ..core.generator import alterego_mapping, alterego_records
    from ..session import session_of
    sess = session_of(trainRDD)
    records = alterego_records(sess, alterego_mapping(privatemap_tool, sess, extended_simRDD, private))
    ctx = getattr(trainRDD, "context", None)
    return ctx.parallelize(records) if ctx is not None else LocalRDD(records)


def map_to_dict(rdd):
    """{source item: target item}, later records overwrite earlier (assist.py:210-215)."""
    return dict((line[1], line[0]) for line in records_of(rdd))


def load_parameter(path):
    """assist.py:228-231 (safe_load: plain yaml.load raises on PyYAML >= 6)."""
    import yaml
    with open(path, "rb") as f:
        return yaml.safe_load(f)


def write_to_disk(results, out_dict, path):
    """assist.py:234-244."""
    import yaml
    out_folder = join(path, "runs", str(int(time.time())))
    makedirs(out_folder)
    out_dict["result"] = results
    with open(join(out_folder, "info.yaml"), "w") as f:
        f.write(yaml.dump(out_dict, default_flow_style=False))


# downstream recommender stages on the AlterEgo profile (assist.py:153-207): see core/recommender.py
from ..core.recommender import (recommender_calculate_sim_pipeline, recommender_privacy_pipeline,  # noqa: E402,F401
                                recommender_prediction_pipeline)
