from .params import load_params
from .params import dump_params
from .train import train
from .train import fit_parameter
from .train import train_epoch
from .train import evaluate
