"""Host-side mirror of the reference's stage classes (xmap/core/*.py) plus, as
the north-star asks, the five pipeline functions (which the reference keeps in
xmap.utils.assist; its xmap/core/__init__.py is empty)."""
from .als import ALS, MatrixFactorizationModel, Rating
from .baselinerClean import BaselinerClean
from .baselinerSplit import BaselinerSplit
from .baselinerSim import BaselinerSim
from .extender import ExtendSim
from .generator import Generator
from .recommender import (RecommenderSim, RecommenderPrivacy, RecommenderPrediction,
                          recommender_calculate_sim_pipeline, recommender_privacy_pipeline,
                          recommender_prediction_pipeline, recommend_top_n)
from ..utils.assist import (baseliner_clean_data_pipeline, baseliner_split_data_pipeline,
                            baseliner_calculate_sim_pipeline, extender_pipeline, generator_pipeline)

__all__ = ["BaselinerClean", "BaselinerSplit", "BaselinerSim", "ExtendSim", "Generator",
           "RecommenderSim", "RecommenderPrivacy", "RecommenderPrediction", "recommender_calculate_sim_pipeline",
           "recommender_privacy_pipeline", "recommender_prediction_pipeline", "recommend_top_n",
           "baseliner_clean_data_pipeline", "baseliner_split_data_pipeline",
           "baseliner_calculate_sim_pipeline", "extender_pipeline", "generator_pipeline",
           "ALS", "MatrixFactorizationModel", "Rating"]
