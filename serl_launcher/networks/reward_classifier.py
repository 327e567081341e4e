"""reference networks/reward_classifier.py -> serl_b200 (plus the lazy device batch and train step of the example's training loop)."""
from serl_b200.networks.reward_classifier import (ClassifierState, create_classifier, load_classifier_func,  # noqa: F401
                                                   sample_classifier_batch, train_step)
