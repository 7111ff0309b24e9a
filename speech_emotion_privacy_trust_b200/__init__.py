"""B200-native (sm_100a) speech feature extraction + cloak / gradient-reversal path.

Host layer over libsept_b200.so (C ABI in include/sept.h).  Sub-modules:
    extraction      ragged-batch log-mel / MFCC
    normalization   per-speaker statistics, normalisation, training-window assembly
    augmentation    class-balance noise augmentation of the training windows
    cloak_ops       autograd functions of the fused cloak + gradient-reversal kernels
    wave_cloak      the waveform-domain cloak: learned periodic noise on the raw audio of a ragged batch
    parallel        utterance sharding and the data-parallel gradient all-reduce
    dropin/         modules with the reference's names and signatures
There is no CPU compute path: everything above fails loudly without the CUDA library and a CUDA device.
"""
__version__ = "0.1.0"
