"""Held-out evaluation of the two-domain experiment on the device: the test split of ingest_arrays against the item-based
predictions (MAE) and the top-N lists (precision, recall, NDCG, MAP at n, coverage) of the AlterEgo profile.

    A = ingest.ingest_arrays(clean_source, clean_target, split_tool, path_source, path_target, False)
    ev = evaluate.evaluate(A, sim_tool, extend_tool, generator, private_gen, rec_sim_tool, privacy_tool, private_rec)

The tools are the facade chain's (BaselinerSim, ExtendSim, Generator, RecommenderSim, RecommenderPrivacy), so every
parameter, private mode and seed means what it means there, and the predictions, the MAE and the lists equal those of
clean_split_pipeline -> ... -> recommender_prediction_pipeline / recommend_top_n (with the time zone at UTC: the
facade turns times into local datetimes and back with timegm).  Every array stays on the device; no Python object is
made per record.  The reference has no ranking metrics: their definitions are in DESIGN.md section 3.6.

    ev = evaluate.evaluate_als(A, rank=10, iterations=5, lambda_=0.01)          # the MLlib-ALS baseline

evaluate_als runs the same held-out evaluation on explicit ALS (als.py, DESIGN.md section 3.8), trained on every
training record of both domains or on the AlterEgo profile."""
import math
from dataclasses import dataclass

import torch

from . import als as ALS
from . import generate as G
from . import ingest as I
from . import recsim as RS
from .core.baselinerSim import SimHandle
from .core.generator import alterego_mapping
from .core.recommender import ProfileState, recommender_privacy_pipeline
from .session import Session


@dataclass
class Evaluation:
    """evaluate's result.  Held-out pairs follow A.test_* order; evaluated users are ids of A.all_uids."""
    mae_nodecay: float           # None when no pair was predicted
    mae_decay: float
    pred_nodecay: torch.Tensor   # f64 [n_test] bounded prediction, -1 where the pair was skipped
    pred_decay: torch.Tensor
    users: torch.Tensor          # int64 [n_eval] all_uids index of each evaluated user
    metrics: RS.RankMetrics      # per evaluated user, the means and the coverage
    top: RS.TopN                 # rows indexed by train user; items index profile_items
    profile_items: torch.Tensor  # int64: train item index of every profile item (profile item index = position)
    n: int
    counts: dict
    stage_ms: dict               # device time per stage when events were passed, else None


def _alterego_profile(A, sim_tool, extend_tool, generator, private_gen, timer):
    """Train arrays -> similarity -> X-SIM -> mapping -> the AlterEgo profile in the facade's list order (target records
    in training order, then the synthetic ones): (user, item, rating, ts, profile_items, synthetic record count).
    Profile items are numbered by rank among the items present, as the facade's np.unique over id strings does (the
    private selection draws per item index); users keep the train numbering (only their order matters)."""
    dev = A.user.device
    if sim_tool.method not in ("cosine", "adjust_cosine"):
        raise ValueError("unknown similarity method %r" % (sim_tool.method,))
    if A.train_user_of is None or A.train_item_of is None:
        raise ValueError("the arrays carry no train index maps (train_user_of / train_item_of)")
    with timer("session"):
        sess = Session(I.encoded(A), dev, user=A.user, item=A.item, rating=A.rating, meta=A.meta)
    with timer("similarity_xsim"):
        xs = extend_tool.extend(SimHandle(sess, sim_tool.method, sim_tool.num_atleast))
    with timer("alterego"):
        mapping = alterego_mapping(generator, sess, xs, private_gen)
        ou, oi, orr, ot = G.build_alterego(sess.layout, torch.arange(sess.layout.nnz, device=dev), mapping)
        keep = A.meta.has_T[A.item.long()]
        pu = torch.cat([A.user.long()[keep], ou.long()])
        pi = torch.cat([A.item.long()[keep], oi.long()])
        pr = torch.cat([A.rating[keep], orr])
        pt = torch.floor(torch.cat([A.ts[keep], A.ts[ot.long()]])).long()      # timegm of the facade's datetimes
        profile_items, pi = torch.unique(pi, return_inverse=True)
    return pu, pi, pr, pt, profile_items, int(ou.numel())


def _profile_index(A, profile_items):
    """The profile index of every train item, -1 outside the profile."""
    prof_of = torch.full((len(A.iids),), -1, dtype=torch.int64, device=A.user.device)
    prof_of[profile_items] = torch.arange(int(profile_items.numel()), device=A.user.device)
    return prof_of


def _test_pairs(A, profile_items, in_prof_user):
    """The held-out pairs in train numbering and then in profile numbering: (tu, tpi, untrained, no_profile)."""
    tu = A.train_user_of[A.test_user.long()].long()
    ti = A.train_item_of[A.test_item.long()].long()
    untrained = (tu < 0) | (ti < 0)
    tpi = torch.where(untrained, -1, _profile_index(A, profile_items)[ti.clamp(min=0)])
    no_profile = ~untrained & ((tpi < 0) | ~in_prof_user[tu.clamp(min=0)])
    return tu, tpi, untrained, no_profile


def _scatter_predictions(counts, ok, preds, fill, untrained, no_profile, predicted, **skipped):
    """preds (values of the held-out pairs ok) spread over every held-out pair, `fill` elsewhere; the pair counts go
    into counts, the model's own reasons to skip a pair in `skipped`."""
    n_test = int(untrained.numel())
    out = []
    for p in preds:
        full = torch.full((n_test,), fill, dtype=torch.float64, device=p.device)
        full[ok] = p
        out.append(full)
    counts.update(test_pairs=n_test, predicted=predicted, skipped_untrained=int(untrained.sum()),
                  skipped_no_profile=int(no_profile.sum()), **skipped)
    return out


def _eval_users(A, threshold):
    """The relevant held-out records (rating >= threshold, of a test user) and the evaluated users, the trained test
    users with one, ascending by all_uids index: (rel, is_test, has_rel, trained, users, run = their train index)."""
    dev = A.user.device
    n_test = int(A.test_user.numel())
    rel = torch.ones(n_test, dtype=torch.bool, device=dev) if threshold is None else A.test_rating >= threshold
    is_test = torch.zeros(len(A.all_uids), dtype=torch.bool, device=dev)
    is_test[torch.from_numpy(A.test_users).to(dev)] = True
    rel &= is_test[A.test_user.long()]
    has_rel = torch.zeros(len(A.all_uids), dtype=torch.bool, device=dev)
    has_rel[A.test_user.long()[rel]] = True
    trained = A.train_user_of >= 0
    users = torch.nonzero(has_rel & trained).flatten()          # ascending all_uids index
    run = A.train_user_of[users].long()
    return rel, is_test, has_rel, trained, users, run


def _relevant_csr(A, rel, users, profile_items):
    """Each evaluated user's relevant items in profile numbering, sorted and unique: (rel_ptr, code).  An item outside
    the profile gets a code past every profile item."""
    dev = A.user.device
    n_items = int(profile_items.numel())
    q_of = torch.full((len(A.all_uids),), -1, dtype=torch.int64, device=dev)
    q_of[users] = torch.arange(int(users.numel()), device=dev)
    rq = q_of[A.test_user.long()[rel]]
    keep_r = rq >= 0
    rq, ri_all = rq[keep_r], A.test_item.long()[rel][keep_r]
    rti = A.train_item_of[ri_all].long()
    code = torch.where(rti >= 0, _profile_index(A, profile_items)[rti.clamp(min=0)], -1)
    code = torch.where(code >= 0, code, n_items + ri_all)
    key = torch.unique(rq * (n_items + len(A.all_iids)) + code)
    rq, code = key // (n_items + len(A.all_iids)), key % (n_items + len(A.all_iids))
    rel_ptr = torch.zeros(int(users.numel()) + 1, dtype=torch.int64, device=dev)
    rel_ptr[1:] = torch.cumsum(torch.bincount(rq, minlength=int(users.numel())), 0)
    return rel_ptr, code


def evaluate(A, sim_tool, extend_tool, generator, private_gen, rec_sim_tool, privacy_tool, private_rec, n=10,
             threshold=None, alpha=0.03, events=None):
    """Train arrays -> similarity -> X-SIM -> mapping -> AlterEgo profile -> item-kNN (or user-kNN when rec_sim_tool's
    method is "cosine_user" / "adjust_cosine_user", DESIGN.md 3.9), then the held-out MAE of the test pairs and the
    top-n accuracy of the test users.  private_gen / private_rec: the generator's private mode and
    the private neighbour selection, as generator_pipeline's and recommender_privacy_pipeline's flags.  threshold: a
    held-out record is relevant when its rating >= threshold (None: every one).  events: optional dict that receives
    CUDA-event pairs per stage; their times are then in stage_ms."""
    timer = I._Timer(events)
    counts = {}

    # ---- AlterEgo profile, in the facade's list order: target records in training order, then the synthetic ones ----
    pu, pi, pr, pt, profile_items, n_synth = _alterego_profile(A, sim_tool, extend_tool, generator, private_gen, timer)
    counts["profile_records"], counts["synthetic_records"] = int(pu.numel()), n_synth
    ev = _eval_users(A, threshold)
    users, run = ev[-2:]
    in_prof_user = torch.bincount(pu, minlength=len(A.uids)) > 0
    chain = _user_based if "cosine_user" in rec_sim_tool.method else _item_based
    top, pred0, pred1, mae0, mae1, listable = chain(A, pu, pi, pr, pt, profile_items, in_prof_user, run, rec_sim_tool,
                                                    privacy_tool, private_rec, n, alpha, timer, counts)
    metrics = _rank_tail(A, ev, top, profile_items, listable, n, timer, counts,
                         eval_users_without_profile=int((~in_prof_user[run]).sum()))
    return Evaluation(mae0, mae1, pred0, pred1, users, metrics, top, profile_items, n, counts, timer.stage_ms())


def _item_based(A, pu, pi, pr, pt, profile_items, in_prof_user, run, rec_sim_tool, privacy_tool, private_rec, n,
                alpha, timer, counts):
    """The item-based chain of evaluate: item-kNN, the prediction of the held-out pairs and the top-n of the train
    users `run`.  Returns (top, pred0, pred1, mae0, mae1, which profile items can be listed)."""
    n_users = len(A.uids)
    with timer("item_knn"):
        state = ProfileState.from_arrays(pu, pi, pr, pt, A.uids, A.iids[profile_items.cpu().numpy()])
        recommender_privacy_pipeline(privacy_tool, rec_sim_tool.calculate_sim(state), private_rec)
        knn, nb = state.knn, state.nb
    with timer("prediction"):
        tu, tpi, untrained, no_profile = _test_pairs(A, profile_items, in_prof_user)
        ok = torch.nonzero(~untrained & ~no_profile).flatten()
        p0, p1, mae0, mae1 = RS.predict(pu, pi, pr, pt, n_users, knn, nb, tu[ok], tpi[ok], A.test_rating[ok], alpha)
    n_pred = int((p0 >= 0).sum())
    pred0, pred1 = _scatter_predictions(counts, ok, (p0, p1), -1.0, untrained, no_profile, n_pred,
                                        skipped_no_neighbours=int(ok.numel()) - n_pred)
    with timer("top_n"):
        top = RS.top_n(pu, pi, pr, pt, n_users, knn, nb, n, alpha=alpha, users=run)
    return top, pred0, pred1, mae0, mae1, nb.len > 0


def _user_based(A, pu, pi, pr, pt, profile_items, in_prof_user, run, rec_sim_tool, privacy_tool, private_rec, n,
                alpha, timer, counts):
    """The user-based chain of evaluate (DESIGN.md 3.9).  Users are renumbered by rank among the profile's users, as the
    facade's np.unique over id strings numbers them (ties and private draws go by that index); only the rows of the
    users with a held-out pair or a list to rank are computed.  Returns what _item_based returns, top's rows by train
    user."""
    from . import usersim as US
    dev = A.user.device
    n_users, n_items = len(A.uids), int(profile_items.numel())
    profile_users, qu = torch.unique(pu, return_inverse=True)
    n_pu = int(profile_users.numel())
    q_of = torch.full((n_users,), -1, dtype=torch.int64, device=dev)
    q_of[profile_users] = torch.arange(n_pu, device=dev)
    with timer("prediction_pairs"):
        tu, tpi, untrained, no_profile = _test_pairs(A, profile_items, in_prof_user)
        ok = torch.nonzero(~untrained & ~no_profile).flatten()
        run_q = q_of[run]
        query = torch.unique(torch.cat([q_of[tu[ok]], run_q[run_q >= 0]]))
    with timer("user_knn"):
        state = ProfileState.from_arrays(qu, pi, pr, pt, A.uids[profile_users.cpu().numpy()],
                                         A.iids[profile_items.cpu().numpy()])
        state.query_users = query
        recommender_privacy_pipeline(privacy_tool, rec_sim_tool.calculate_sim(state), private_rec)
        knn, nb = state.knn, state.nb
    with timer("prediction"):
        p0, p1, mae0, mae1 = US.predict(qu, pi, pr, pt, n_items, knn, nb, q_of[tu[ok]], tpi[ok], A.test_rating[ok],
                                        alpha)
    n_pred = int((p0 >= 0).sum())
    pred0, pred1 = _scatter_predictions(counts, ok, (p0, p1), -1.0, untrained, no_profile, n_pred,
                                        skipped_no_neighbours=int(ok.numel()) - n_pred)
    with timer("top_n"):
        t = US.top_n(qu, pi, pr, pt, n_pu, n_items, knn, nb, n, alpha=alpha, users=run_q[run_q >= 0])
        idx, score, ln = RS.empty_lists(n_users, n, dev)
        idx[profile_users], score[profile_users], ln[profile_users] = t.idx, t.score, t.len
        top = RS.TopN(idx, score, ln, t.visits, t.candidates, t.warp_users, t.cta_users)
    # every profile item can be listed for a user without a record on it
    return top, pred0, pred1, mae0, mae1, torch.ones(n_items, dtype=torch.bool, device=dev)


def _rank_tail(A, ev, top, profile_items, listable, n, timer, counts, **model_count):
    """rank_metrics of the evaluated users' lists against their relevant held-out items (ev: _eval_users; listable:
    which profile items a list can hold, the catalogue), and the counts that do not depend on the model, with
    model_count (the one that does) in its place among them."""
    rel, is_test, has_rel, trained, users, run = ev
    n_items = int(profile_items.numel())
    with timer("rank_metrics"):
        rel_ptr, code = _relevant_csr(A, rel, users, profile_items)
        catalogue = int(listable.sum())
        metrics = RS.rank_metrics(top, run, rel_ptr, code, n, catalogue=catalogue)
        reachable = torch.zeros(int(code.numel()), dtype=torch.bool, device=code.device)
        in_prof = code < n_items
        reachable[in_prof] = listable[code[in_prof]]
    counts.update(eval_users=int(users.numel()), **model_count, test_users_untrained=int((has_rel & ~trained).sum()),
                  test_users_without_relevant=int(len(A.test_users)) - int((has_rel & is_test).sum()),
                  relevant_items=int(code.numel()), unreachable_items=int((~reachable).sum()),
                  catalogue_items=catalogue)
    return metrics


@dataclass
class AlsEvaluation:
    """evaluate_als's result.  Held-out pairs follow A.test_* order; evaluated users are ids of A.all_uids."""
    mae: float                   # mean |rating - score| over the predicted pairs (None when none was)
    mae_bounded: float           # the same with the score rounded as rs_bound_rating does: int(x + 0.5) within [0, 5]
    pred: torch.Tensor           # f64 [n_test] raw score, NaN where the pair was skipped
    users: torch.Tensor          # int64 [n_eval] all_uids index of each evaluated user
    metrics: RS.RankMetrics
    top: ALS.AlsTopN             # rows indexed by train user; items index profile_items
    model: ALS.AlsModel          # users in train numbering, items in profile numbering
    profile_items: torch.Tensor  # int64: train item index of every trained item (trained item index = position)
    train_user: torch.Tensor     # int64: the records the model was trained on
    train_item: torch.Tensor     # int64, profile numbering
    train_rating: torch.Tensor   # f64
    n: int
    counts: dict
    stage_ms: dict               # device time per stage when events were passed, else None


def evaluate_als(A, rank=10, iterations=5, lambda_=0.01, seed=None, alterego=None, n=10, threshold=None, events=None):
    """Explicit ALS (als.train, DESIGN.md 3.8) on the training split, then the held-out MAE of the test pairs and the
    top-n accuracy of the test users, as evaluate reports them for item-kNN.
    alterego: None trains on every training record of both domains (the baseline: a test user keeps its source-domain
    records, so every trained test user has factors); (sim_tool, extend_tool, generator, private_gen) builds the
    AlterEgo profile as evaluate does and trains on it ("X-MAP + ALS").
    mae uses the raw score, as MLlib's predict returns it; mae_bounded rounds it as the item-kNN prediction does.
    The lists cover the target-domain items with factors, minus the user's training records; the catalogue is those
    items.  threshold / events: as in evaluate; with events the model also carries its per-half-step kernel times."""
    dev = A.user.device
    timer = I._Timer(events)
    counts = {}
    if A.train_user_of is None or A.train_item_of is None:
        raise ValueError("the arrays carry no train index maps (train_user_of / train_item_of)")
    n_users = len(A.uids)
    if alterego is None:
        pu, pi, pr = A.user.long(), A.item.long(), A.rating
        profile_items = torch.arange(len(A.iids), device=dev)
    else:
        sim_tool, extend_tool, generator, private_gen = alterego
        pu, pi, pr, _, profile_items, n_synth = _alterego_profile(A, sim_tool, extend_tool, generator, private_gen,
                                                                  timer)
        counts["synthetic_records"] = n_synth
    n_items = int(profile_items.numel())
    counts["train_records"] = int(pu.numel())

    with timer("als_train"):
        model = ALS.train(pu, pi, pr, n_users, n_items, rank, iterations, lambda_, seed=seed, device=dev,
                          events={} if events is not None else None)

    with timer("prediction"):
        tu, tpi, untrained, no_profile = _test_pairs(A, profile_items, model.user_count > 0)
        no_factors = ~untrained & ~no_profile & (model.item_count[tpi.clamp(min=0)] == 0)
        ok = torch.nonzero(~untrained & ~no_profile & ~no_factors).flatten()
        p = ALS.predict(model, tu[ok], tpi[ok])
        mae = mae_b = None
        if int(ok.numel()):
            tr = A.test_rating[ok]
            bounded = torch.clamp(torch.trunc(p + 0.5), 0, 5)
            mae = math.fsum((tr - p).abs().cpu().tolist()) / int(ok.numel())
            mae_b = math.fsum((tr - bounded).abs().cpu().tolist()) / int(ok.numel())
    pred, = _scatter_predictions(counts, ok, (p,), float("nan"), untrained, no_profile, int(ok.numel()),
                                 skipped_no_factors=int(no_factors.sum()))

    ev = _eval_users(A, threshold)
    users, run = ev[-2:]
    with timer("top_n"):
        listable = A.meta.has_T[profile_items] & (model.item_count > 0)
        top = ALS.top_n(model, n, pu, pi, candidates=torch.nonzero(listable).flatten(), users=run)
    metrics = _rank_tail(A, ev, top, profile_items, listable, n, timer, counts,
                         eval_users_without_factors=int((model.user_count[run] == 0).sum()))
    return AlsEvaluation(mae, mae_b, pred, users, metrics, top, model, profile_items, pu, pi, pr, n, counts,
                         timer.stage_ms())
