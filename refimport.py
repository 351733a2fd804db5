"""Import the UNMODIFIED reference (skycrapers/TecoGAN-PyTorch) from the checkout named by the
environment variable TECOGAN_REFERENCE (its root directory, the one holding codes/).

Used only where the reference itself is the subject: oracle/gen_golden.py (writes the fixtures under
tests/golden), `bench.py --impl reference`/`--impl eager-gpu` (optional) and the training workloads of
bench.py (which run the reference's own training loop); the product package and the test suite never
import it.  Recipe = SURVEY.md section 9: no reference file is edited; the modules this image lacks
(skimage / IPython behind metrics/__init__, lmdb behind data/) are stubbed in sys.modules and two
renamed library symbols are aliased.
"""
import os
import sys
import types

ENV = 'TECOGAN_REFERENCE'


def reference_codes_dir():
    root = os.environ.get(ENV)
    codes = os.path.join(root, 'codes') if root else None
    if codes and os.path.isfile(os.path.join(codes, 'models', 'networks', 'tecogan_nets.py')):
        return codes
    return None


def available():
    return reference_codes_dir() is not None


def _prepare():
    codes = reference_codes_dir()
    if codes is None:
        raise ImportError(f'the reference is not available: set {ENV} to the root of a TecoGAN-PyTorch checkout')
    if codes not in sys.path:
        sys.path.insert(0, codes)
    if 'metrics' not in sys.modules or getattr(sys.modules['metrics'], '__refimport__', None) != codes:
        m = types.ModuleType('metrics')
        m.__path__ = [os.path.join(codes, 'metrics')]    # skip metrics/__init__ (LPIPS -> skimage/IPython)
        m.create_metric_calculator = lambda opt: None    # only needed to import main.py
        m.__refimport__ = codes
        sys.modules['metrics'] = m
    sys.modules.setdefault('lmdb', types.ModuleType('lmdb'))
    import scipy.signal
    import scipy.signal.windows
    if not hasattr(scipy.signal, 'gaussian'):            # utils/data_utils.py:15 uses the removed alias
        scipy.signal.gaussian = scipy.signal.windows.gaussian
    return codes


def import_generator():
    """-> (FRNet class, net_utils module, data_utils module) of the reference"""
    _prepare()
    from models.networks.tecogan_nets import FRNet
    from utils import net_utils, data_utils
    return FRNet, net_utils, data_utils


def import_models():
    """-> the reference's `models` package (VSRModel / VSRGANModel / define_generator) and `main`"""
    _prepare()
    import models
    import models.networks
    import models.vsr_model
    import main
    return models, main


def root_dir():
    codes = reference_codes_dir()
    return None if codes is None else os.path.dirname(codes)


def stub_pretrained_vgg19(seed=0):
    """codes/models/networks/vgg_nets.py:11 asks torchvision for vgg19(pretrained=True); there is no
    network here, so the perceptual-loss extractor gets seeded random weights of the same architecture
    (same FLOPs and memory traffic -- this only matters for benchmarks and integration tests)."""
    import torch
    import torchvision
    real = torchvision.models.vgg19

    def vgg19(pretrained=False, **kw):
        g = torch.random.get_rng_state()
        torch.manual_seed(seed)
        try:
            return real(weights=None)
        finally:
            torch.random.set_rng_state(g)

    if getattr(torchvision.models.vgg19, '__name__', '') != 'vgg19' or not hasattr(torchvision.models.vgg19, '_stub'):
        vgg19._stub = True
        torchvision.models.vgg19 = vgg19


def training_opt(model='tecogan', device='cuda:0', dist=False, rank=0, world_size=1, nb=10):
    """The reference's own training YAML (experiments_BD/{TecoGAN,FRVSR}/*_REDS_4xSR_2GPU/train.yml) as the
    `opt` dict its models take, with the data/checkpoint paths the offline box does not have removed."""
    import yaml
    sub = {'tecogan': ('TecoGAN', 'TecoGAN_REDS_4xSR_2GPU'), 'frvsr': ('FRVSR', 'FRVSR_REDS_4xSR_2GPU')}[model]
    path = os.path.join(root_dir(), 'experiments_BD', sub[0], sub[1], 'train.yml')
    opt = yaml.safe_load(open(path))
    opt['model']['generator']['load_path'] = None
    opt['model']['generator']['nb'] = nb
    if 'discriminator' in opt['model']:
        opt['model']['discriminator']['load_path'] = None
    opt.update({'device': device, 'dist': dist, 'is_train': True, 'rank': rank, 'world_size': world_size})
    opt['train']['ckpt_dir'] = '/tmp'
    return opt


def build_training_model(opt, define_generator=None):
    """VSRModel / VSRGANModel of the reference for `opt`; define_generator (e.g. tecogan_b200's) replaces
    the reference's generator factory for the duration of the construction."""
    models, _ = import_models()
    import models.vsrgan_model as vg
    import models.vsr_model as vm
    cls = vg.VSRGANModel if opt['model']['name'].lower() == 'tecogan' else vm.VSRModel
    saved = (vm.define_generator, vg.define_generator)
    if define_generator is not None:
        vm.define_generator = vg.define_generator = define_generator
    try:
        if cls is vg.VSRGANModel:
            stub_pretrained_vgg19()
        return cls(opt)
    finally:
        vm.define_generator, vg.define_generator = saved
