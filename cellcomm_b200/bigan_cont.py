"""Drop-in for the reference's `src/bigan_cont.py`: the continuous-code BiGAN the trainer
actually uses (ContinuousCellBiGan :44-56), with the wider generator / encoder scaled by
gene_size (:7-41) and the discriminator inherited from bigan_classify."""
import numpy as np

try:
    from .bigan_basic import BasicBiGan
    from .bigan_classify import ClassifyCellBiGan
    from . import engine as _engine
    from .models import NetModel
except ImportError:  # imported as top-level modules (PYTHONPATH=src style)
    from bigan_basic import BasicBiGan
    from bigan_classify import ClassifyCellBiGan
    from cellcomm_b200 import engine as _engine
    from cellcomm_b200.models import NetModel


def _build_generator(encoding_size, gene_size):
    return NetModel(_engine.cont_generator_graph(encoding_size, gene_size), "G",
                    [("gen_encoding_in", "z"), ("gen_random_in", "r")])


def _build_encoder(encoding_size, gene_size):
    return NetModel(_engine.cont_encoder_graph(encoding_size, gene_size), "E",
                    [("enc_cell_in", "cell")])


class ContinuousCellBiGan(ClassifyCellBiGan):
    VARIANT = "cont"

    def __init__(self, encoding_size, gene_size, **kwargs):
        super().__init__(
            encoding_size, gene_size,
            generator_factory=_build_generator,
            encoder_factory=_build_encoder,
            **kwargs
        )

    def random_encoding_vector(self, batch_size):
        """tf.random.uniform(shape=(batch_size, encoding_size), 0, 1) (reference :52-53)."""
        return self._prior_rng.random((batch_size, self.encoding_size), dtype=np.float32)

    def trainings_encoding_prediction(self, cell_data):
        return self.encoding_prediction(cell_data)

    # a continuous code has no classes: compare_cells uses one group and random encodings
    _comparison_groups = BasicBiGan._comparison_groups
    _comparison_encodings = BasicBiGan._comparison_encodings
