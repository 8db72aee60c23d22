"""Generate tests/golden/*.npz from the UNMODIFIED reference (/root/reference).

Run in the build container only (the GPU box has no reference checkout):

    PYTHONDONTWRITEBYTECODE=1 python -m oracle.make_golden

Every fixture stores the inputs next to the reference's outputs, so the tests
need neither the reference nor this script; the full-size and deflationSeed
fixtures, which would pass 1 MB with them, store outputs only and the tests
regenerate their inputs from the seeded generators of oracle/synth.py.
Quantities with an arbitrary phase / sign (eigenvectors, beamforming vectors,
Watson modes) are stored as produced AND compared phase-invariantly by the tests.
"""
import os

import numpy as np

from . import ref_shim, synth

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                   'tests', 'golden')


def _cacgmm_case(ref, name, y, init, iterations, **kw):
    T = ref.distribution.CACGMMTrainer
    model = T().fit(y, initialization=init, iterations=iterations, **kw)
    aff, q = model.predict(
        y, return_quadratic_form=True,
        source_activity_mask=kw.get('source_activity_mask'))
    out = dict(
        y=y, init=init, iterations=iterations,
        weight=model.weight,
        eigenvectors=model.cacg.covariance_eigenvectors,
        eigenvalues=model.cacg.covariance_eigenvalues,
        covariance=model.cacg.covariance,
        affiliation=aff, quadratic_form=q,
        log_likelihood=model.log_likelihood(y),
    )
    for k, v in kw.items():
        out['kw_' + k] = np.asarray(v if v is not False else 0)
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
    return model


def make_cacgmm(ref):
    # structured mixture, D=4 K=2 (config C1 scaled down)
    y, _ = synth.structured_stft(6, 60, 4, 2, seed=1)
    init = synth.init_affiliation(6, 2, 60, seed=7)
    _cacgmm_case(ref, 'cacgmm_d4k2', y, init, 8)
    # noise input, D=8 K=3 (config C2 scaled down)
    y = synth.noise_stft(4, 70, 8, seed=0)
    init = synth.init_affiliation(4, 3, 70, seed=7)
    _cacgmm_case(ref, 'cacgmm_d8k3', y, init, 6)
    # structured D=8 K=3: near-singular covariances, exercises the floor
    y, _ = synth.structured_stft(3, 90, 8, 3, seed=2)
    init = synth.init_affiliation(3, 3, 90, seed=3)
    _cacgmm_case(ref, 'cacgmm_d8k3_structured', y, init, 10)
    # option variants on a small D=3 K=2 problem (dims of the reference's tests)
    y, _ = synth.structured_stft(3, 50, 3, 2, seed=5)
    init = synth.init_affiliation(3, 2, 50, seed=11)
    rng = np.random.RandomState(4)
    sal = rng.uniform(0.1, 1.0, size=(3, 50))
    sam = rng.uniform(size=(3, 2, 50)) > 0.2
    sam[:, 0, :] |= ~sam[:, 1, :]  # at least one class active per frame
    _cacgmm_case(ref, 'cacgmm_opt_saliency', y, init, 5, saliency=sal)
    _cacgmm_case(ref, 'cacgmm_opt_mask', y, init, 5,
                 source_activity_mask=sam)
    _cacgmm_case(ref, 'cacgmm_opt_trace', y, init, 5, covariance_norm='trace')
    _cacgmm_case(ref, 'cacgmm_opt_nonorm', y, init, 5, covariance_norm=False)
    _cacgmm_case(ref, 'cacgmm_opt_w2', y, init, 5, weight_constant_axis=-2)
    _cacgmm_case(ref, 'cacgmm_opt_eps0', y, init, 5, affiliation_eps=0.,
                 eigenvalue_floor=1e-6)
    # broadcast initialisation (singleton independent dim), cacgmm.py:221-228
    _cacgmm_case(ref, 'cacgmm_opt_bcast', y, init[:1], 5)
    # warm start from a model: 3 + 2 iterations, cacgmm.py:229-234
    T = ref.distribution.CACGMMTrainer
    m3 = T().fit(y, initialization=init, iterations=3)
    m5 = T().fit(y, initialization=m3, iterations=2)
    np.savez_compressed(
        os.path.join(OUT, 'cacgmm_warm.npz'), y=y, init=init,
        w3=m3.weight, V3=m3.cacg.covariance_eigenvectors,
        l3=m3.cacg.covariance_eigenvalues,
        w5=m5.weight, cov5=m5.cacg.covariance,
        l5=m5.cacg.covariance_eigenvalues)


def make_cacgmm_coupled(ref):
    """Frequency-tied weights and inline permutation alignment (cacgmm.py:252-278)."""
    pa = ref.permutation_alignment
    y, _ = synth.structured_stft(65, 60, 4, 2, seed=21)
    init = synth.init_affiliation(65, 2, 60, seed=5)
    _cacgmm_case(ref, 'cacgmm_tied_time', y, init, 5, weight_constant_axis=(-3,))
    _cacgmm_case(ref, 'cacgmm_tied', y, init, 5, weight_constant_axis=(-3, -1))
    # saliency together with tied weights, and tied weights with a batch dim in front of the bins
    sal = np.random.RandomState(9).uniform(0.2, 1.0, size=(65, 60))
    _cacgmm_case(ref, 'cacgmm_tied_time_saliency', y, init, 4, weight_constant_axis=(-3,), saliency=sal)
    _cacgmm_case(ref, 'cacgmm_tied_saliency', y, init, 4, weight_constant_axis=(-3, -1), saliency=sal)
    yb = np.stack([y[:33], synth.structured_stft(33, 60, 4, 2, seed=22)[0]])
    _cacgmm_case(ref, 'cacgmm_tied_batch', yb, np.stack([init[:33], init[32:]]), 4, weight_constant_axis=(-3,))
    al = pa.DHTVPermutationAlignment(stft_size=128, segment_start=20, segment_width=20, segment_shift=5,
                                     main_iterations=5, sub_iterations=2)
    T = ref.distribution.CACGMMTrainer
    model = T().fit(y, initialization=init, iterations=5, weight_constant_axis=(-3,),
                    inline_permutation_aligner=al)
    np.savez_compressed(
        os.path.join(OUT, 'cacgmm_inline_pa.npz'), y=y, init=init, iterations=5,
        plan=np.asarray(al.alignment_plan), weight=model.weight,
        eigenvalues=model.cacg.covariance_eigenvalues, covariance=model.cacg.covariance,
        affiliation=model.predict(y))


def make_cacg_steps(ref):
    """Single E / M step pieces on fixed model parameters."""
    rng = np.random.RandomState(21)
    F, K, D, T = 3, 3, 5, 40
    y = synth.noise_stft(F, T, D, seed=9)
    z = ref.cacg.normalize_observation(y)
    cov = synth.pos_def_hermitian(F, K, D, D, seed=3)
    m = ref.cacg.ComplexAngularCentralGaussian.from_covariance(
        cov.copy(), eigenvalue_floor=1e-10)
    log_pdf, q = m._log_pdf(z[..., None, :, :])
    w = rng.uniform(size=(F, K, 1))
    w /= w.sum(-2, keepdims=True)
    aff = ref.mixture_model_utils.log_pdf_to_affiliation(
        w, log_pdf, affiliation_eps=1e-10)
    m2 = ref.cacg.ComplexAngularCentralGaussianTrainer()._fit(
        z[..., None, :, :], aff, q)
    np.savez_compressed(
        os.path.join(OUT, 'cacg_steps.npz'), y=y, z=z, cov=cov,
        V=m.covariance_eigenvectors, lam=m.covariance_eigenvalues,
        log_pdf=log_pdf, q=q, w=w, aff=aff,
        fit_cov=m2.covariance, fit_lam=m2.covariance_eigenvalues)


def make_cwmm(ref):
    T = ref.distribution.CWMMTrainer
    cases = {
        'cwmm_d6k4': (synth.structured_stft(4, 120, 6, 4, seed=6)[0], 4, 6),
        'cwmm_d4k2': (synth.structured_stft(5, 80, 4, 2, seed=8)[0], 2, 7),
    }
    for name, (y, K, it) in cases.items():
        F, N, D = y.shape
        init = synth.init_affiliation(F, K, N, seed=13)
        tr = T()
        model = tr.fit(y, initialization=init, iterations=it)
        aff = model.predict(y)
        np.savez_compressed(
            os.path.join(OUT, name + '.npz'), y=y, init=init, iterations=it,
            weight=model.weight, mode=model.complex_watson.mode,
            concentration=model.complex_watson.concentration,
            affiliation=aff)
    # the spline itself (the concentration look-up table is model state)
    for D in (4, 6, 8):
        tr = ref.complex_watson.ComplexWatsonTrainer(D)
        lam = np.concatenate([
            [0, 1 / D, 1 / D + 1e-4, 0.9599999, 1],
            np.linspace(1 / D - 0.01, 1.0, 200)])
        np.savez_compressed(
            os.path.join(OUT, f'cw_spline_d{D}.npz'), D=D, lam=lam,
            kappa=tr.hypergeometric_ratio_inverse(lam),
            kappa_grid=np.linspace(0, 500, 101),
            log_norm=ref.complex_watson.ComplexWatson.log_norm_1f1(
                np.linspace(0, 500, 101), D))


def make_cwmm_coupled(ref):
    """CWMMTrainer with frequency-tied weights and the inline permutation alignment (cwmm.py:76-240)."""
    T = ref.distribution.CWMMTrainer
    pa = ref.permutation_alignment
    y = synth.structured_stft(65, 60, 4, 2, seed=21)[0]
    F, N, D = y.shape
    K = 2
    init = synth.init_affiliation(F, K, N, seed=13)
    for name, axis, inline in (('cwmm_tied_time', (-3,), False), ('cwmm_tied', (-3, -1), False),
                               ('cwmm_inline_pa', (-3,), True)):
        al = pa.DHTVPermutationAlignment(stft_size=128, segment_start=20, segment_width=20, segment_shift=5,
                                         main_iterations=5, sub_iterations=2) if inline else None
        model = T().fit(y, initialization=init, iterations=4, weight_constant_axis=axis,
                        inline_permutation_aligner=al)
        out = dict(y=y, init=init, iterations=4, weight=model.weight, mode=model.complex_watson.mode,
                   concentration=model.complex_watson.concentration, affiliation=model.predict(y))
        if inline:
            out['plan'] = np.asarray(al.alignment_plan)
        np.savez_compressed(os.path.join(OUT, name + '.npz'), **out)
    sal = np.random.RandomState(9).uniform(0.2, 1.0, size=(F, N))
    model = T().fit(y, initialization=init, iterations=4, weight_constant_axis=(-3,), saliency=sal)
    np.savez_compressed(os.path.join(OUT, 'cwmm_tied_time_saliency.npz'), y=y, init=init, iterations=4, saliency=sal,
                        weight=model.weight, mode=model.complex_watson.mode,
                        concentration=model.complex_watson.concentration, affiliation=model.predict(y))


def make_permutation(ref):
    pa = ref.permutation_alignment
    rng = np.random.RandomState(31)
    out = {}
    # (a) default 512-point plan on a synthetic permuted mask, F=257
    for tag, stft_size, K, T in (('a', 512, 3, 40), ('b', 1024, 2, 30)):
        F = stft_size // 2 + 1
        proto = rng.uniform(size=(K, 1, T)) ** 4
        mask = proto + 0.35 * rng.uniform(size=(K, F, T))
        mask /= mask.sum(0, keepdims=True)
        perm = np.stack([rng.permutation(K) for _ in range(F)], axis=1)
        mask = mask[perm, np.arange(F)]
        al = pa.DHTVPermutationAlignment.from_stft_size(stft_size)
        mapping = al.calculate_mapping(mask.copy())
        out[f'{tag}_mask'] = mask
        out[f'{tag}_plan'] = np.asarray(al.alignment_plan)
        out[f'{tag}_mapping'] = mapping
        out[f'{tag}_aligned'] = al.apply_mapping(mask, mapping)
    # (c) custom small plan, K=4, pure noise mask (many near ties)
    K, F, T = 4, 65, 25
    mask = rng.uniform(size=(K, F, T))
    mask /= mask.sum(0, keepdims=True)
    al = pa.DHTVPermutationAlignment(
        stft_size=128, segment_start=20, segment_width=20, segment_shift=5,
        main_iterations=5, sub_iterations=2)
    out['c_mask'] = mask
    out['c_plan'] = np.asarray(al.alignment_plan)
    out['c_mapping'] = al.calculate_mapping(mask.copy())
    # the non-default options of DHTV (:133-163) on mask (a): every metric with both assignments
    mask = out['a_mask']
    for metric in ('cos', 'multiply', 'euclidean'):
        for algorithm in ('greedy', 'optimal'):
            al = pa.DHTVPermutationAlignment(
                stft_size=512, segment_start=70, segment_width=100, segment_shift=20, main_iterations=20,
                sub_iterations=2, similarity_metric=metric, algorithm=algorithm)
            out[f'opt_{metric}_{algorithm}'] = al.calculate_mapping(mask.copy())
    # greedy assignment known answer, permutation_alignment.py:475-508
    sm = np.array([[11, 10, 0], [4, 5, 10], [6, 0, 5]])
    out['score'] = sm
    out['score_greedy'] = pa._mapping_from_score_matrix(sm, 'greedy')
    np.savez_compressed(os.path.join(OUT, 'permutation.npz'), **out)


def make_permutation_greedy_oracle(ref):
    """GreedyPermutationAlignment / OraclePermutationAlignment / _mapping_from_score_matrix
    (permutation_alignment.py:458-786) on a permuted synthetic mask and on pure noise."""
    pa = ref.permutation_alignment
    rng = np.random.RandomState(32)
    out = {}
    K, F, T = 3, 65, 40
    proto = rng.uniform(size=(K, 1, T)) ** 4
    clean = proto + 0.5 * rng.uniform(size=(K, F, T))
    clean /= clean.sum(0, keepdims=True)
    perm = np.stack([rng.permutation(K) for _ in range(F)], axis=1)
    out['mask'] = clean[perm, np.arange(F)]
    out['reference_mask'] = clean
    noise = rng.uniform(size=(4, 33, 20))
    out['noise'] = noise / noise.sum(0, keepdims=True)
    out['noise_reference'] = rng.uniform(size=(4, 33, 20))
    for metric in ('cos', 'euclidean', 'multiply'):
        out[f'greedy_{metric}'] = pa.GreedyPermutationAlignment(metric).calculate_mapping(out['mask'])
        out[f'greedy_noise_{metric}'] = pa.GreedyPermutationAlignment(metric).calculate_mapping(out['noise'])
        out[f'scores_{metric}'] = getattr(pa._ScoreMatrix, metric)(out['noise'], out['noise_reference'])
        for alg in ('greedy', 'optimal'):
            al = pa.OraclePermutationAlignment(metric, alg)
            out[f'oracle_{metric}_{alg}'] = al.calculate_mapping(out['mask'], out['reference_mask'])
            out[f'oracle_noise_{metric}_{alg}'] = al.calculate_mapping(out['noise'], out['noise_reference'])
    sm = np.array([[11, 10, 0], [4, 5, 10], [6, 0, 5]])  # doctest, :475-508
    out['score'] = sm
    out['score_greedy'] = pa._mapping_from_score_matrix(sm, 'greedy')
    out['score_optimal'] = pa._mapping_from_score_matrix(sm, 'optimal')
    np.savez_compressed(os.path.join(OUT, 'permutation_greedy_oracle.npz'), **out)


def make_beamformer(ref):
    bf = ref.beamformer
    F, D, T, K = 9, 6, 80, 3
    rng = np.random.RandomState(41)
    Y = np.swapaxes(synth.structured_stft(F, T, D, K, seed=12)[0], -1, -2)
    Y = np.ascontiguousarray(Y)
    mask = rng.uniform(size=(F, K, T))
    mask /= mask.sum(1, keepdims=True)
    psd = bf.get_power_spectral_density_matrix(Y, mask)
    psd_nonorm = bf.get_power_spectral_density_matrix(Y, mask,
                                                      normalize=False)
    psd_single = bf.get_power_spectral_density_matrix(Y, mask[:, 0])
    psd_nomask = bf.get_power_spectral_density_matrix(Y)
    target, noise = psd[:, 0], psd[:, 1] + psd[:, 2]
    pca = bf.get_pca_vector(target)
    mvdr = bf.get_mvdr_vector(pca, noise)
    gev = bf._get_gev_vector(target, noise)
    souden, ref_ch = bf.get_mvdr_vector_souden(target, noise,
                                               return_ref_channel=True)
    ban = bf.blind_analytic_normalization(gev, noise)
    applied = bf.apply_beamforming_vector(gev, Y)
    np.savez_compressed(
        os.path.join(OUT, 'beamformer.npz'), Y=Y, mask=mask, psd=psd,
        psd_nonorm=psd_nonorm, psd_single=psd_single, psd_nomask=psd_nomask,
        target=target, noise=noise, pca=pca, mvdr=mvdr, gev=gev,
        souden=souden, ref_channel=ref_ch, ban=ban, applied=applied)


def make_bf_wrapper(ref):
    import importlib
    bw = importlib.import_module('pb_bss.extraction.beamformer_wrapper')
    g = np.load(os.path.join(OUT, 'beamformer.npz'))
    target, noise = g['target'], g['noise']
    out = dict(target=target, noise=noise)
    names = ['pca', 'pca+mvdr', 'scaled_gev_atf+mvdr', 'mvdr_souden', 'mvdr_souden+ban',
             'rank1_pca+mvdr_souden', 'rank1_gev+mvdr_souden+ban', 'gev', 'gev+ban',
             'rank1_pca+gev', 'ch1']
    for n in names:
        out['bf_' + n] = np.asarray(bw.get_bf_vector(n, target.copy(), noise.copy()))
    out['rank1_pca'] = bw.get_pca_rank_one_estimate(target.copy())
    out['rank1_gev'] = bw.get_gev_rank_one_estimate(target.copy(), noise.copy())
    np.savez_compressed(os.path.join(OUT, 'bf_wrapper.npz'), **out)


def make_full_size(ref):
    """BASELINE.json configs 2 and 4 at FULL size, outputs only (the seeded inputs are regenerated by the tests):
    the fitted model on every bin and the affiliations of every bin at every 8th frame.  Every fixture file stays
    below 1 MB: the model and the affiliations go to separate files, and the Hermitian covariance is stored as its
    upper triangle (np.triu_indices order, diagonal included)."""
    T = ref.distribution.CACGMMTrainer
    for name, gen in (('c2_full_noise', lambda: synth.noise_stft(513, 500, 8, seed=0)),
                      ('c2_full_structured', lambda: synth.structured_stft(513, 500, 8, 3, seed=21)[0])):
        y = gen()
        init = synth.init_affiliation(513, 3, 500, seed=7)
        model = T().fit(y, initialization=init, iterations=100)
        aff = model.predict(y)
        cov = model.cacg.covariance
        iu = np.triu_indices(cov.shape[-1])
        np.savez_compressed(
            os.path.join(OUT, name + '.npz'), iterations=100,
            weight=model.weight, eigenvalues=model.cacg.covariance_eigenvalues,
            covariance_triu=cov[..., iu[0], iu[1]],
            log_likelihood=model.log_likelihood(y))
        np.savez_compressed(os.path.join(OUT, name + '_affiliation.npz'), affiliation_8=aff[..., ::8])
    y = synth.noise_stft(257, 1000, 6, seed=4)
    init = synth.init_affiliation(257, 4, 1000, seed=7)
    model = ref.distribution.CWMMTrainer().fit(y, initialization=init, iterations=50)
    aff = model.predict(y)
    np.savez_compressed(
        os.path.join(OUT, 'c4_full_noise.npz'), iterations=50, weight=model.weight,
        mode=model.complex_watson.mode, concentration=model.complex_watson.concentration)
    np.savez_compressed(os.path.join(OUT, 'c4_full_noise_affiliation.npz'), affiliation_8=aff[..., ::8])


def make_gcacgmm(ref):
    """Integrated model GCACGMM (gcacgmm.py:38-333): spherical / diagonal Gaussians over embeddings, weight layouts,
    the inline pairing of spatial and spectral classes."""
    import pb_bss.distribution.gcacgmm as G
    F, T, D, E, K = 20, 70, 4, 5, 3
    y, labels = synth.structured_stft(F, T, D, K, seed=41)
    rng = np.random.RandomState(5)
    centers = rng.randn(K, E) * 2.0
    emb = centers[labels] + 0.7 * rng.randn(F, T, E)           # (F, T, E): class-dependent embedding clouds
    init = synth.init_affiliation(F, K, T, seed=3)
    sal = rng.uniform(0.3, 1.0, size=(F, T))
    cases = {
        'spherical': dict(),
        'diagonal_kt': dict(covariance_type='diagonal', weight_constant_axis=(-3,)),
        'spherical_k_inline': dict(weight_constant_axis=(-3, -1), inline_permutation_alignment=True),
        'spherical_sal_weights': dict(saliency=sal, spatial_weight=0.7, spectral_weight=1.3),
    }
    out = dict(y=y, embedding=emb, init=init, saliency=sal)
    for name, kw in cases.items():
        model = G.GCACGMMTrainer().fit(y, emb, initialization=init, iterations=4, **kw)
        out[f'{name}_weight'] = np.asarray(model.weight)
        out[f'{name}_mean'] = model.gaussian.mean
        out[f'{name}_gcov'] = model.gaussian.covariance
        out[f'{name}_eigenvalues'] = model.cacg.covariance_eigenvalues
        out[f'{name}_covariance'] = model.cacg.covariance
        out[f'{name}_affiliation'] = model.predict(y, emb)
    np.savez_compressed(os.path.join(OUT, 'gcacgmm.npz'), **out)
    # the same problem with the von Mises-Fisher spectral model (vmfcacgmm.py:34-301)
    import pb_bss.distribution.vmfcacgmm as V
    vcases = {
        'vmf': dict(),
        'vmf_kt_inline': dict(weight_constant_axis=(-3,), inline_permutation_alignment=True, max_concentration=50),
        'vmf_sal': dict(saliency=sal, spatial_weight=0.6, spectral_weight=1.2, weight_constant_axis=(-3, -1)),
    }
    vout = dict(y=y, embedding=emb, init=init, saliency=sal)
    for name, kw in vcases.items():
        model = V.VMFCACGMMTrainer().fit(y, emb, initialization=init, iterations=4, **kw)
        vout[f'{name}_weight'] = np.asarray(model.weight)
        vout[f'{name}_mean'] = model.vmf.mean
        vout[f'{name}_concentration'] = model.vmf.concentration
        vout[f'{name}_eigenvalues'] = model.cacg.covariance_eigenvalues
        vout[f'{name}_covariance'] = model.cacg.covariance
        vout[f'{name}_affiliation'] = model.predict(y, emb)
    np.savez_compressed(os.path.join(OUT, 'vmfcacgmm.npz'), **vout)


def make_initializer(ref):
    """pb_bss.initializer: iid draws after np.random.seed(0), flag, deflationSeed (deflation.py:6-89)."""
    import pb_bss.initializer as RI
    out = {}
    Y = np.ones([4, 5, 3])
    for name in ('uniform_normalized', 'dirichlet_uniform', 'one_hot'):
        for pf in (False, True):
            np.random.seed(0)
            out[f'{name}_{int(pf)}'] = np.array(getattr(RI.iid, name)(Y, 2, permutation_free=pf))
    np.random.seed(0)
    out['dirichlet_a3'] = np.array(RI.iid.dirichlet(np.ones([2, 7, 3]), 3, alpha=3))
    out['flag_2'] = np.array(RI.deterministic.flag(Y, 2, permutation_free=True))
    out['flag_4_min'] = np.array(RI.deterministic.flag(np.ones([1, 5, 3]), 4, minimum=0.1, permutation_free=True))
    # the inputs are not stored (the file would pass 1 MB): the test regenerates them from the same seeds
    y = synth.structured_stft(257, 60, 4, 3, seed=17)[0]
    out['deflation_pf'] = RI.deflation.deflationSeed(y, 3, permutation_free=True)
    out['deflation_nopf'] = RI.deflation.deflationSeed(y, 3, permutation_free=False, neighbors=3)
    sal = np.random.RandomState(2).uniform(0.1, 1, size=(257, 60))
    out['deflation_with_sal'] = RI.deflation.deflationSeed(y, 2, saliencies=sal, eps=1e-3)
    np.savez_compressed(os.path.join(OUT, 'initializer.npz'), **out)


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = ref_shim.load()
    import sys
    if len(sys.argv) > 1 and sys.argv[1] == 'full':
        make_full_size(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'initializer':
        make_initializer(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'permutation':
        make_permutation(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'gcacgmm':
        make_gcacgmm(ref)
        return
    if len(sys.argv) > 1 and sys.argv[1] == 'coupled':
        make_cacgmm_coupled(ref)
        make_cwmm_coupled(ref)
        return
    make_cacgmm(ref)
    make_cacgmm_coupled(ref)
    make_cacg_steps(ref)
    make_cwmm(ref)
    make_cwmm_coupled(ref)
    make_permutation(ref)
    make_permutation_greedy_oracle(ref)
    make_beamformer(ref)
    make_bf_wrapper(ref)
    make_initializer(ref)
    make_gcacgmm(ref)
    make_full_size(ref)
    total = 0
    for n in sorted(os.listdir(OUT)):
        s = os.path.getsize(os.path.join(OUT, n))
        total += s
        print(f'{n:36s} {s:8d} B')
    print('total', total)


if __name__ == '__main__':
    main()
