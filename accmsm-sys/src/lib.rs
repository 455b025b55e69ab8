//! `accmsm-sys`: the Rust side of the drop-in boundary of libaccmsm.so (include/accmsm.h).
//!
//! * [`ffi`] -- every entry point of the C-ABI, generated from the header (tools/gen_sys_bindings.py);
//! * safe wrappers over the memory images ark-ff / ark-ec 0.2 use (SURVEY.md App. A.4): a field element is the
//!   `BigInteger256([u64; 4])` inside `Fp256` (Montgomery form, little-endian limbs), an affine point is `x`, `y` and the
//!   `infinity` flag.  `GroupAffine` is `repr(Rust)`: points are marshalled FIELD BY FIELD, never transmuted.  Slices of
//!   `Fp256<P>` are passed as they lie in memory: `Fp256<P>` is `BigInteger256` + `PhantomData` (size and alignment of
//!   `[u64; 4]`, checked by a const assertion below), and `into_repr()` happens on the device.
//!
//! The wrappers are generic over the two curves the library implements through [`GpuCurve`]; `ark-poly-commit` calls
//! them from `PedersenCommitment::commit`, `InnerProductArgPC::{cm_commit, check, open}` (integration/ark-poly-commit.patch).
//! `ark-accumulation` itself is untouched: `AccumulationScheme`, the key / index types and the curve generics stay.
#![allow(clippy::missing_safety_doc)]

pub mod ffi;

use ark_ec::short_weierstrass_jacobian::GroupAffine;
use ark_ec::SWModelParameters;
use ark_ff::{BigInteger256, Fp256, Fp256Parameters, Zero};
use std::ffi::CStr;
use std::os::raw::c_int;
use std::sync::{Arc, Mutex, Once};

/// A curve of the Pallas / Vesta cycle as the library numbers them (`curve`: 0 = Pallas, 1 = Vesta; the scalar field of
/// one is the base field of the other, `field`: 0 = Fp, 1 = Fq).
pub trait GpuCurve: SWModelParameters {
    const CURVE_ID: c_int;
    const SCALAR_FIELD_ID: c_int;
}
// implemented for ark_pallas::PallasParameters (0, 1) and ark_vesta::VestaParameters (1, 0) by the crate that owns
// those types' dependency (ark-poly-commit's patch adds the two one-line impls; orphan rules keep them out of here).

#[derive(Debug, Clone)]
pub struct GpuError {
    pub code: c_int,
    pub message: String,
}
impl std::fmt::Display for GpuError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "accmsm error {}: {}", self.code, self.message)
    }
}
impl std::error::Error for GpuError {}
pub type Result<T> = std::result::Result<T, GpuError>;

/// One context: a single GPU or a group of GPUs of one box.  Calls are serialised inside the library; the handle is
/// `Send + Sync`.  There is no CPU fallback: construction fails without a CUDA device.
pub struct Context {
    raw: *mut ffi::accmsm_ctx,
}
unsafe impl Send for Context {}
unsafe impl Sync for Context {}

impl Context {
    pub fn new(device: i32) -> Result<Arc<Self>> {
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { ffi::accmsm_init(&mut raw, device as c_int) };
        if rc != 0 {
            return Err(GpuError { code: rc, message: strerror(rc) });
        }
        Ok(Arc::new(Context { raw }))
    }
    /// `accmsm_init_multi`: keys are sharded by point range across `devices` inside the library; every call below spans them.
    pub fn new_multi(devices: &[i32]) -> Result<Arc<Self>> {
        let devs: Vec<c_int> = devices.iter().map(|&d| d as c_int).collect();
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { ffi::accmsm_init_multi(&mut raw, devs.as_ptr(), devs.len() as c_int) };
        if rc != 0 {
            return Err(GpuError { code: rc, message: strerror(rc) });
        }
        Ok(Arc::new(Context { raw }))
    }
    /// Process-wide context: `ACCMSM_DEVICES=0,1,2,3` selects a device group, default is device 0.
    pub fn global() -> Arc<Self> {
        static INIT: Once = Once::new();
        static mut GLOBAL: Option<Arc<Context>> = None;
        unsafe {
            INIT.call_once(|| {
                let devs: Vec<i32> = std::env::var("ACCMSM_DEVICES")
                    .ok()
                    .map(|s| s.split(',').filter_map(|t| t.trim().parse().ok()).collect())
                    .unwrap_or_default();
                let ctx = if devs.len() > 1 { Context::new_multi(&devs) } else { Context::new(*devs.first().unwrap_or(&0)) };
                GLOBAL = Some(ctx.expect("accmsm: no CUDA device (there is no CPU fallback)"));
            });
            GLOBAL.as_ref().unwrap().clone()
        }
    }
    pub fn raw(&self) -> *mut ffi::accmsm_ctx {
        self.raw
    }
    fn check(&self, rc: c_int) -> Result<()> {
        if rc == 0 {
            return Ok(());
        }
        let detail = unsafe { CStr::from_ptr(ffi::accmsm_last_error(self.raw)) }.to_string_lossy().into_owned();
        Err(GpuError { code: rc, message: format!("{} ({})", strerror(rc), detail) })
    }
}
impl Drop for Context {
    fn drop(&mut self) {
        unsafe { ffi::accmsm_destroy(self.raw) }
    }
}

fn strerror(rc: c_int) -> String {
    unsafe { CStr::from_ptr(ffi::accmsm_strerror(rc)) }.to_string_lossy().into_owned()
}

// Fp256<P> must be exactly the four limbs: slices of field elements cross the boundary as they lie in memory.
const _: () = assert!(std::mem::size_of::<BigInteger256>() == 32 && std::mem::align_of::<BigInteger256>() == 8);
fn limbs_of<P: Fp256Parameters>(v: &[Fp256<P>]) -> *const u64 {
    debug_assert_eq!(std::mem::size_of::<Fp256<P>>(), 32);
    v.as_ptr() as *const u64
}
fn fe_from_limbs<P: Fp256Parameters>(l: &[u64]) -> Fp256<P> {
    // the limbs ARE the Montgomery image: Fp256::new, not from_repr
    Fp256::<P>::new(BigInteger256([l[0], l[1], l[2], l[3]]))
}
/// Ties a curve's base field to its limbs (both Pallas and Vesta have 255-bit `Fp256` base fields).  Implemented next to
/// [`GpuCurve`] for the two parameter sets: `base_limbs(x) = (x.0).0`, `base_from_limbs(l) = Fp256::new(BigInteger256(l))`
/// (the limbs ARE the Montgomery image: `new`, not `from_repr`).
pub trait GpuBase: SWModelParameters {
    fn base_limbs(x: &Self::BaseField) -> [u64; 4];
    fn base_from_limbs(l: &[u64]) -> Self::BaseField;
}
fn affine_from<P: GpuBase>(xy: &[u64; 8], inf: u8) -> GroupAffine<P> {
    if inf != 0 {
        return GroupAffine::<P>::zero();      // (0, 1, infinity = true), what the library writes too
    }
    GroupAffine::<P>::new(P::base_from_limbs(&xy[0..4]), P::base_from_limbs(&xy[4..8]), false)
}

/// A commitment key resident in HBM (`accmsm_register_bases`): `ck.generators` (and, when present, the hiding generator as
/// the LAST base, so `PedersenCommitment::commit(ck, elems, Some(r))` is one pass).  Registered once at `trim` / `index` time
/// (src/ipa_pc_as/mod.rs:507-513, src/hp_as/mod.rs:640-641); the window table is built with it.
pub struct GpuKey {
    ctx: Arc<Context>,
    handle: u64,
    n_generators: usize,
    hiding_index: Option<usize>,
    lock: Mutex<()>,
}
impl GpuKey {
    pub fn register<P: GpuCurve + GpuBase>(ctx: &Arc<Context>, generators: &[GroupAffine<P>], hiding: Option<&GroupAffine<P>>) -> Result<Self> {
        let n = generators.len() + hiding.is_some() as usize;
        let mut xy = Vec::<u64>::with_capacity(n * 8);
        let mut inf = Vec::<u8>::with_capacity(n);
        for g in generators.iter().chain(hiding.into_iter()) {
            xy.extend_from_slice(&P::base_limbs(&g.x));
            xy.extend_from_slice(&P::base_limbs(&g.y));
            inf.push(g.infinity as u8);
        }
        let mut handle = 0u64;
        ctx.check(unsafe { ffi::accmsm_register_bases(ctx.raw, P::CURVE_ID, xy.as_ptr(), inf.as_ptr(), n, &mut handle) })?;
        ctx.check(unsafe { ffi::accmsm_precompute_bases(ctx.raw, handle, 0) })?;
        Ok(GpuKey { ctx: ctx.clone(), handle, n_generators: generators.len(), hiding_index: hiding.map(|_| generators.len()), lock: Mutex::new(()) })
    }
    pub fn len(&self) -> usize {
        self.n_generators
    }
    pub fn is_empty(&self) -> bool {
        self.n_generators == 0
    }

    /// `VariableBaseMSM::multi_scalar_mul(&bases[..n], &scalars[..n]).into_affine()` with scalars given as field elements
    /// (the form `cm_commit` / `PedersenCommitment::commit` hold them in).  ark-ec truncates to the shorter slice.
    pub fn msm<P: GpuCurve + GpuBase, S: Fp256Parameters>(&self, scalars: &[Fp256<S>]) -> Result<GroupAffine<P>> {
        let n = scalars.len().min(self.n_generators);
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let _g = self.lock.lock().unwrap();
        self.ctx.check(unsafe { ffi::accmsm_msm(self.ctx.raw, self.handle, 0, n, limbs_of(scalars), 1, xy.as_mut_ptr(), &mut inf) })?;
        Ok(affine_from::<P>(&xy, inf))
    }
    /// The literal ark-ec signature: scalars as `BigInteger256` (canonical).
    pub fn msm_bigint<P: GpuCurve + GpuBase>(&self, scalars: &[BigInteger256]) -> Result<GroupAffine<P>> {
        let n = scalars.len().min(self.n_generators);
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        self.ctx.check(unsafe { ffi::accmsm_msm(self.ctx.raw, self.handle, 0, n, scalars.as_ptr() as *const u64, 0, xy.as_mut_ptr(), &mut inf) })?;
        Ok(affine_from::<P>(&xy, inf))
    }
    /// `PedersenCommitment::commit(ck, elems, randomizer)` / `cm_commit(key, scalars, Some(h), Some(r))`.
    pub fn commit<P: GpuCurve + GpuBase, S: Fp256Parameters>(&self, elems: &[Fp256<S>], randomizer: Option<Fp256<S>>) -> Result<GroupAffine<P>> {
        let n = elems.len().min(self.n_generators);
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        let r = randomizer.map(|r| (r.0).0);
        let (hi, rp) = match (&r, self.hiding_index) {
            (Some(r), Some(h)) => (h, r.as_ptr()),
            (Some(_), None) => return Err(GpuError { code: ffi::ACCMSM_E_ARG, message: "commit with a randomizer needs a key registered with its hiding generator".into() }),
            _ => (0, std::ptr::null()),
        };
        self.ctx.check(unsafe { ffi::accmsm_commit(self.ctx.raw, self.handle, n, limbs_of(elems), hi, rp, xy.as_mut_ptr(), &mut inf) })?;
        Ok(affine_from::<P>(&xy, inf))
    }
    /// k commitments over the same key in shared passes (hp_as::decide: src/hp_as/mod.rs:910-918; NARK: r1cs_nark/mod.rs:216-218).
    pub fn msm_batch<P: GpuCurve + GpuBase, S: Fp256Parameters>(&self, vectors: &[&[Fp256<S>]]) -> Result<Vec<GroupAffine<P>>> {
        let k = vectors.len();
        let n = vectors.iter().map(|v| v.len()).min().unwrap_or(0).min(self.n_generators);
        let mut flat = Vec::<u64>::with_capacity(k * n * 4);
        for v in vectors {
            flat.extend_from_slice(unsafe { std::slice::from_raw_parts(limbs_of(&v[..n]), n * 4) });
        }
        let (mut xy, mut inf) = (vec![0u64; 8 * k], vec![0u8; k]);
        self.ctx.check(unsafe { ffi::accmsm_msm_batch(self.ctx.raw, self.handle, 0, n, k, flat.as_ptr(), 1, xy.as_mut_ptr(), inf.as_mut_ptr()) })?;
        Ok((0..k).map(|j| { let mut a = [0u64; 8]; a.copy_from_slice(&xy[8 * j..8 * j + 8]); affine_from::<P>(&a, inf[j]) }).collect())
    }
    /// Tail of `IpaPC::check_individual_opening_challenges` (= AS `decide`, src/ipa_pc_as/mod.rs:836-845):
    /// accept iff `cm_commit(comm_key, h.compute_coeffs()) == proof.final_comm_key`; h(X) never leaves the device.
    pub fn ipa_check_final_key<P: GpuCurve + GpuBase, S: Fp256Parameters>(&self, challenges: &[Fp256<S>], final_comm_key: &GroupAffine<P>) -> Result<bool> {
        let mut exp = [0u64; 8];
        exp[..4].copy_from_slice(&P::base_limbs(&final_comm_key.x));
        exp[4..].copy_from_slice(&P::base_limbs(&final_comm_key.y));
        let mut accept: c_int = 0;
        self.ctx.check(unsafe {
            ffi::accmsm_ipa_check_final_key(self.ctx.raw, self.handle, limbs_of(challenges), challenges.len() as c_int, exp.as_ptr(),
                                            final_comm_key.infinity as u8, &mut accept, std::ptr::null_mut(), std::ptr::null_mut())
        })?;
        Ok(accept != 0)
    }
    /// `ASForHadamardProducts::decide` (src/hp_as/mod.rs:894-925): product on the device, three commitments in one pass.
    pub fn hp_decide<P: GpuCurve + GpuBase, S: Fp256Parameters>(&self, a: &[Fp256<S>], b: &[Fp256<S>], randomness: Option<[Fp256<S>; 3]>,
                                                                 comms: [&GroupAffine<P>; 3]) -> Result<bool> {
        let n = a.len().min(b.len()).min(self.n_generators);
        let mut exp = [0u64; 24];
        let mut exp_inf = [0u8; 3];
        for (j, c) in comms.iter().enumerate() {
            exp[8 * j..8 * j + 4].copy_from_slice(&P::base_limbs(&c.x));
            exp[8 * j + 4..8 * j + 8].copy_from_slice(&P::base_limbs(&c.y));
            exp_inf[j] = c.infinity as u8;
        }
        let r: Option<Vec<u64>> = randomness.map(|r| r.iter().flat_map(|x| (x.0).0.to_vec()).collect());
        let mut accept: c_int = 0;
        self.ctx.check(unsafe {
            ffi::accmsm_hp_decide(self.ctx.raw, self.handle, limbs_of(a), limbs_of(b), n, self.hiding_index.unwrap_or(0),
                                  r.as_ref().map_or(std::ptr::null(), |r| r.as_ptr()), exp.as_ptr(), exp_inf.as_ptr(), &mut accept,
                                  std::ptr::null_mut(), std::ptr::null_mut())
        })?;
        Ok(accept != 0)
    }
    pub fn handle(&self) -> u64 {
        self.handle
    }
    pub fn context(&self) -> &Arc<Context> {
        &self.ctx
    }
}
impl Drop for GpuKey {
    fn drop(&mut self) {
        unsafe { ffi::accmsm_release_bases(self.ctx.raw, self.handle) };
    }
}

/// `IpaPC::open_individual_opening_challenges` as a device session (the host keeps the sponge):
/// `begin` -> k x { `round` -> (l, r); xi = sponge(..); `fold(xi, xi^-1)` } -> `finish` -> (final_comm_key, c).
pub struct IpaOpenSession<'k> {
    key: &'k GpuKey,
    id: u64,
    finished: bool,
}
impl<'k> IpaOpenSession<'k> {
    /// `h_prime` is passed as `xi_0` when the key holds the hiding generator (`h' = xi_0 * h` then rides in each round's MSM).
    pub fn begin<S: Fp256Parameters>(key: &'k GpuKey, coeffs: &[Fp256<S>], log_d: usize, point: Fp256<S>, xi0: Fp256<S>) -> Result<Self> {
        let h = key.hiding_index.ok_or(GpuError { code: ffi::ACCMSM_E_ARG, message: "the opening needs the hiding generator in the key".into() })?;
        let mut id = 0u64;
        key.ctx.check(unsafe { ffi::accmsm_ipa_open_begin(key.ctx.raw, key.handle, limbs_of(coeffs), coeffs.len(), log_d as c_int, (point.0).0.as_ptr(), std::ptr::null(), &mut id) })?;
        key.ctx.check(unsafe { ffi::accmsm_ipa_open_use_hiding_generator(key.ctx.raw, id, h, (xi0.0).0.as_ptr()) })?;
        Ok(IpaOpenSession { key, id, finished: false })
    }
    /// zk opening (`MakeZK::Enabled`): begin without xi_0, which upstream squeezes from `C'` only after the hiding step:
    /// `begin_zk` -> `hide` -> hiding_comm; alpha = sponge(C, z, v, hiding_comm); `hiding_challenge(alpha)`;
    /// `C' = C + alpha hiding_comm - (r + alpha rho) s` and xi_0 on the host; `use_hiding_generator(xi_0)`; then the rounds.
    pub fn begin_zk<S: Fp256Parameters>(key: &'k GpuKey, coeffs: &[Fp256<S>], log_d: usize, point: Fp256<S>) -> Result<Self> {
        let mut id = 0u64;
        key.ctx.check(unsafe { ffi::accmsm_ipa_open_begin(key.ctx.raw, key.handle, limbs_of(coeffs), coeffs.len(), log_d as c_int, (point.0).0.as_ptr(), std::ptr::null(), &mut id) })?;
        Ok(IpaOpenSession { key, id, finished: false })
    }
    /// The random polynomial (<= 2^log_d coefficients) is shifted on the device to vanish at the point and committed:
    /// returns `hiding_comm = cm_commit(comm_key, hiding', Some(s), Some(rho))` with s the key's base `s_index`.
    pub fn hide<P: GpuCurve + GpuBase, S: Fp256Parameters>(&mut self, hiding: &[Fp256<S>], s_index: usize, rho: Fp256<S>) -> Result<GroupAffine<P>> {
        let (mut xy, mut inf) = ([0u64; 8], 0u8);
        self.key.ctx.check(unsafe {
            ffi::accmsm_ipa_open_hide(self.key.ctx.raw, self.id, limbs_of(hiding), hiding.len(), s_index, (rho.0).0.as_ptr(), xy.as_mut_ptr(), &mut inf)
        })?;
        Ok(affine_from::<P>(&xy, inf))
    }
    /// `P += alpha * hiding'` on the device (enqueued only).
    pub fn hiding_challenge<S: Fp256Parameters>(&mut self, alpha: Fp256<S>) -> Result<()> {
        self.key.ctx.check(unsafe { ffi::accmsm_ipa_open_hiding_challenge(self.key.ctx.raw, self.id, (alpha.0).0.as_ptr()) })
    }
    /// `h' = xi_0 * h` with h the key's base `h_index`; before the first round.
    pub fn use_hiding_generator<S: Fp256Parameters>(&mut self, h_index: usize, xi0: Fp256<S>) -> Result<()> {
        self.key.ctx.check(unsafe { ffi::accmsm_ipa_open_use_hiding_generator(self.key.ctx.raw, self.id, h_index, (xi0.0).0.as_ptr()) })
    }
    pub fn round<P: GpuCurve + GpuBase>(&mut self) -> Result<(GroupAffine<P>, GroupAffine<P>)> {
        let (mut l, mut r, mut li, mut ri) = ([0u64; 8], [0u64; 8], 0u8, 0u8);
        self.key.ctx.check(unsafe { ffi::accmsm_ipa_open_round(self.key.ctx.raw, self.id, l.as_mut_ptr(), &mut li, r.as_mut_ptr(), &mut ri) })?;
        Ok((affine_from::<P>(&l, li), affine_from::<P>(&r, ri)))
    }
    pub fn fold<S: Fp256Parameters>(&mut self, xi: Fp256<S>, xi_inv: Fp256<S>) -> Result<()> {
        self.key.ctx.check(unsafe { ffi::accmsm_ipa_open_fold(self.key.ctx.raw, self.id, (xi.0).0.as_ptr(), (xi_inv.0).0.as_ptr()) })
    }
    /// One call per round of the opening loop: fold with the challenge squeezed from the previous `(l, r)` (its inverse is
    /// computed inside the library, on the host, like upstream's `round_challenge.inverse()`) and run the next round.
    /// `None` when that fold was the last one: call `finish` next.
    pub fn fold_round<P: GpuCurve + GpuBase, S: Fp256Parameters>(&mut self, xi: Fp256<S>) -> Result<Option<(GroupAffine<P>, GroupAffine<P>)>> {
        let (mut l, mut r, mut li, mut ri, mut done) = ([0u64; 8], [0u64; 8], 0u8, 0u8, 0 as c_int);
        self.key.ctx.check(unsafe {
            ffi::accmsm_ipa_open_fold_round(self.key.ctx.raw, self.id, (xi.0).0.as_ptr(), l.as_mut_ptr(), &mut li, r.as_mut_ptr(), &mut ri, &mut done)
        })?;
        Ok(if done != 0 { None } else { Some((affine_from::<P>(&l, li), affine_from::<P>(&r, ri))) })
    }
    pub fn finish<P: GpuCurve + GpuBase, S: Fp256Parameters>(mut self) -> Result<(GroupAffine<P>, Fp256<S>)> {
        let (mut fk, mut c) = ([0u64; 8], [0u64; 4]);
        self.finished = true;
        self.key.ctx.check(unsafe { ffi::accmsm_ipa_open_finish(self.key.ctx.raw, self.id, fk.as_mut_ptr(), c.as_mut_ptr()) })?;
        Ok((affine_from::<P>(&fk, 0), fe_from_limbs::<S>(&c)))
    }
}
impl<'k> Drop for IpaOpenSession<'k> {
    fn drop(&mut self) {
        if !self.finished {
            let (mut fk, mut c) = ([0u64; 8], [0u64; 4]);
            unsafe { ffi::accmsm_ipa_open_finish(self.key.ctx.raw, self.id, fk.as_mut_ptr(), c.as_mut_ptr()) };   // releases the session
        }
    }
}

/// `VariableBaseMSM::multi_scalar_mul(&bases, &scalars).into_affine()` for `m` independent MSMs of equal length over their own,
/// unregistered bases in shared passes of the pipeline: the succinct-check group equations of all inputs and accumulators of
/// one ipa-pc-as prove / verify (src/ipa_pc_as/mod.rs:198-205 inside the loops at :262-270 and :625-640).
pub fn msm_oneshot_batch<P: GpuCurve + GpuBase>(ctx: &Context, bases: &[&[GroupAffine<P>]], scalars: &[&[BigInteger256]]) -> Result<Vec<GroupAffine<P>>> {
    let m = bases.len().min(scalars.len());
    let n = (0..m).map(|j| bases[j].len().min(scalars[j].len())).min().unwrap_or(0);
    let (mut xy, mut inf, mut sc) = (Vec::<u64>::with_capacity(m * n * 8), Vec::<u8>::with_capacity(m * n), Vec::<u64>::with_capacity(m * n * 4));
    for j in 0..m {
        for i in 0..n {
            let g = &bases[j][i];
            xy.extend_from_slice(&P::base_limbs(&g.x)); xy.extend_from_slice(&P::base_limbs(&g.y)); inf.push(g.infinity as u8);
            sc.extend_from_slice(&scalars[j][i].0);
        }
    }
    let (mut out, mut oinf) = (vec![0u64; 8 * m], vec![0u8; m]);
    ctx.check(unsafe { ffi::accmsm_msm_oneshot_batch(ctx.raw, P::CURVE_ID, xy.as_ptr(), inf.as_ptr(), sc.as_ptr(), 0, n, m, out.as_mut_ptr(), oinf.as_mut_ptr()) })?;
    Ok((0..m).map(|j| { let mut a = [0u64; 8]; a.copy_from_slice(&out[8 * j..8 * j + 8]); affine_from::<P>(&a, oinf[j]) }).collect())
}

/// Field-vector kernels of the in-tree loops (src/hp_as/mod.rs:278-285,482-512; src/ipa_pc_as/mod.rs:400).
pub mod vec {
    use super::*;
    pub fn hadamard<S: Fp256Parameters + FieldId>(ctx: &Context, a: &[Fp256<S>], b: &[Fp256<S>]) -> Result<Vec<Fp256<S>>> {
        let n = a.len().min(b.len());
        let mut out = vec![Fp256::<S>::from(0u64); n];
        ctx.check(unsafe { ffi::accmsm_vec_hadamard(ctx.raw, S::FIELD_ID, limbs_of(a), limbs_of(b), n, out.as_mut_ptr() as *mut u64) })?;
        Ok(out)
    }
    pub fn compute_coeffs<S: Fp256Parameters + FieldId>(ctx: &Context, challenges: &[Fp256<S>]) -> Result<Vec<Fp256<S>>> {
        let mut out = vec![Fp256::<S>::from(0u64); 1usize << challenges.len()];
        ctx.check(unsafe { ffi::accmsm_compute_coeffs(ctx.raw, S::FIELD_ID, limbs_of(challenges), challenges.len() as c_int, out.as_mut_ptr() as *mut u64) })?;
        Ok(out)
    }
    /// `field` id of an `Fp256` parameter set (0 = Fp, 1 = Fq)
    pub trait FieldId {
        const FIELD_ID: c_int;
    }
}
