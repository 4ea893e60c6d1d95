//! petal-neighbors API (v0.18) over the B200 engine.  Same public names as the reference
//! (`BallTree`, `VantagePointTree`, `ArrayError`, `distance::{Metric, Euclidean}`), so a
//! dependent crate switches by changing one line of Cargo.toml.  Single-point methods are
//! batches of one; `query_batch` & co. are the additions that let a GPU earn its keep.
//!
//! NOT compiled in the build image (no cargo/rustc there) -- see INTEGRATION.md.
pub mod distance;
mod ffi;

use std::ffi::CStr;
use std::marker::PhantomData;

use ndarray::{Array1, Array2, ArrayBase, ArrayView2, CowArray, Data, Ix1, Ix2};
use thiserror::Error;

pub use distance::Euclidean;
use ffi::Element;

/// The error type for input arrays (reference src/lib.rs:9-16).
#[derive(Debug, Error)]
pub enum ArrayError {
    #[error("array is empty")]
    Empty,
    #[error("array is not contiguous in memory")]
    NotContiguous,
}

fn last_error() -> String {
    unsafe { CStr::from_ptr(ffi::pn_last_error_message()).to_string_lossy().into_owned() }
}

fn check_create(status: i32) -> Result<(), ArrayError> {
    match status {
        ffi::PN_OK => Ok(()),
        ffi::PN_EMPTY => Err(ArrayError::Empty),
        ffi::PN_NOT_CONTIGUOUS => Err(ArrayError::NotContiguous),
        s => panic!("petal_b200 status {s}: {}", last_error()), // internal invariants: the reference uses expect()
    }
}

fn check(status: i32) {
    if status != ffi::PN_OK {
        panic!("petal_b200 status {status}: {}", last_error());
    }
}

struct Handle(*mut ffi::pn_tree);
unsafe impl Send for Handle {}
unsafe impl Sync for Handle {} // queries serialise inside the library
impl Drop for Handle {
    fn drop(&mut self) {
        unsafe { ffi::pn_tree_destroy(self.0) };
    }
}

/// Element strides of a 2-D array as the C ABI wants them, or `None` when a stride is negative
/// (a reversed view): the caller then copies to standard layout first.  Casting a negative `isize`
/// stride with `as usize` would hand the engine a huge positive one.
fn strides<A>(points: &CowArray<'_, A, Ix2>) -> Option<(usize, usize)> {
    let s = points.strides();
    if (points.nrows() > 1 && s[0] < 0) || (points.ncols() > 1 && s[1] < 0) {
        return None;
    }
    let rs = if points.nrows() > 1 { s[0] as usize } else { points.ncols().max(1) };
    let cs = if points.ncols() > 1 { s[1] as usize } else { 1 };
    Some((rs, cs))
}

/// The reference's distance fold zips the two rows and silently truncates to the shorter one
/// (src/distance.rs:26-35).  The C ABI reads exactly `d` elements per query row, so a wrong-sized
/// query would be an out-of-bounds read from safe code: every query method checks first.
fn check_dim(got: usize, want: usize, what: &str) {
    assert!(got == want, "petal_neighbors: {what} has dimension {got}, the tree has {want}");
}

/// Points for `create`: borrowed as they are when the strides are non-negative, otherwise copied
/// to standard layout (the copy only lives for the duration of the call -- the engine keeps its
/// own flattened copy on the device).
fn with_points<A: Element, R>(
    points: &CowArray<'_, A, Ix2>,
    f: impl FnOnce(*const A, usize, usize, usize, usize) -> R,
) -> R {
    let (n, d) = (points.nrows(), points.ncols());
    match strides(points) {
        Some((rs, cs)) => f(points.as_ptr(), n, d, rs, cs),
        None => {
            let dense = points.as_standard_layout();
            f(dense.as_ptr(), n, d, d.max(1), 1)
        }
    }
}

/// Ball tree; the partition is built on the host with the reference's split rule and lives,
/// flattened, in GPU memory.
pub struct BallTree<'a, A, M = Euclidean> {
    handle: Handle,
    n: usize,
    d: usize,
    pub metric: M,
    _p: PhantomData<&'a A>,
}

impl<'a, A: Element> BallTree<'a, A, Euclidean> {
    /// reference src/ball_tree.rs:367-373
    pub fn euclidean<T: Into<CowArray<'a, A, Ix2>>>(points: T) -> Result<Self, ArrayError> {
        Self::new(points, Euclidean::default())
    }

    /// reference src/ball_tree.rs:38-63 (`metric` must be `Euclidean`: the only one on the GPU)
    pub fn new<T: Into<CowArray<'a, A, Ix2>>>(points: T, metric: Euclidean) -> Result<Self, ArrayError> {
        let points: CowArray<'a, A, Ix2> = points.into();
        let (n, d) = (points.nrows(), points.ncols());
        let mut h = std::ptr::null_mut();
        check_create(with_points(&points, |p, n, d, rs, cs| unsafe { A::ball_create(p, n, d, rs, cs, std::ptr::null(), &mut h) }))?;
        Ok(Self { handle: Handle(h), n, d, metric, _p: PhantomData })
    }

    /// reference src/ball_tree.rs:80-86
    pub fn query_nearest<S: Data<Elem = A>>(&self, point: &ArrayBase<S, Ix1>) -> (usize, A) {
        check_dim(point.len(), self.d, "point");
        let q = point.to_owned();
        let (mut i, mut dist) = (0u64, A::zero());
        check(unsafe { A::ball_nearest(self.handle.0, q.as_ptr(), 1, self.d, &mut i, &mut dist) });
        (i as usize, dist)
    }

    /// reference src/ball_tree.rs:102-121
    pub fn query<S: Data<Elem = A>>(&self, point: &ArrayBase<S, Ix1>, k: usize) -> (Vec<usize>, Vec<A>) {
        check_dim(point.len(), self.d, "point");
        if k == 0 {
            return (Vec::new(), Vec::new());
        }
        let q = point.to_owned();
        let mut idx = vec![0u64; k];
        let mut dist = vec![A::zero(); k];
        check(unsafe { A::ball_query(self.handle.0, q.as_ptr(), 1, self.d, k, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        let m = k.min(self.n); // k > n returns n results (the heap never fills)
        (idx[..m].iter().map(|&i| i as usize).collect(), dist[..m].to_vec())
    }

    /// reference src/ball_tree.rs:137-142 (indices ascending)
    pub fn query_radius<S: Data<Elem = A>>(&self, point: &ArrayBase<S, Ix1>, distance: A) -> Vec<usize> {
        check_dim(point.len(), self.d, "point");
        let q = point.to_owned();
        let (offsets, indices) = self.radius_raw(q.as_ptr(), 1, self.d, distance);
        debug_assert_eq!(offsets.len(), 2);
        indices
    }

    /// Batched `query`: row-major `nq x k`; rows padded with (usize::MAX, +inf) when k > n.
    pub fn query_batch(&self, queries: &ArrayView2<A>, k: usize) -> (Array2<usize>, Array2<A>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        let nq = q.nrows();
        let mut idx = vec![0u64; nq * k];
        let mut dist = vec![A::zero(); nq * k];
        check(unsafe { A::ball_query(self.handle.0, q.as_ptr(), nq, self.d, k, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        (
            Array2::from_shape_vec((nq, k), idx.into_iter().map(|i| i as usize).collect()).unwrap(),
            Array2::from_shape_vec((nq, k), dist).unwrap(),
        )
    }

    pub fn query_nearest_batch(&self, queries: &ArrayView2<A>) -> (Array1<usize>, Array1<A>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        let nq = q.nrows();
        let mut idx = vec![0u64; nq];
        let mut dist = vec![A::zero(); nq];
        check(unsafe { A::ball_nearest(self.handle.0, q.as_ptr(), nq, self.d, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        (idx.into_iter().map(|i| i as usize).collect(), Array1::from_vec(dist))
    }

    /// Batched `query_radius`: CSR `(offsets[nq + 1], indices)`.
    pub fn query_radius_batch(&self, queries: &ArrayView2<A>, distance: A) -> (Vec<usize>, Vec<usize>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        self.radius_raw(q.as_ptr(), q.nrows(), self.d, distance)
    }

    fn radius_raw(&self, q: *const A, nq: usize, qs: usize, r: A) -> (Vec<usize>, Vec<usize>) {
        let (mut po, mut pi) = (std::ptr::null_mut::<u64>(), std::ptr::null_mut::<u64>());
        check(unsafe { A::ball_radius(self.handle.0, q, nq, qs, r, &mut po, &mut pi) });
        unsafe {
            let offsets: Vec<usize> = std::slice::from_raw_parts(po, nq + 1).iter().map(|&v| v as usize).collect();
            let total = *offsets.last().unwrap();
            let indices: Vec<usize> = std::slice::from_raw_parts(pi, total).iter().map(|&v| v as usize).collect();
            ffi::pn_free(po.cast());
            ffi::pn_free(pi.cast());
            (offsets, indices)
        }
    }

    /// Every stored point as a query (the loop of the reference's bench, benches/ball_tree.rs:53-59).
    pub fn query_self(&self, k: usize) -> (Array2<usize>, Array2<A>) {
        let mut idx = vec![0u64; self.n * k];
        let mut dist = vec![A::zero(); self.n * k];
        check(unsafe { A::ball_self(self.handle.0, k, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        (
            Array2::from_shape_vec((self.n, k), idx.into_iter().map(|i| i as usize).collect()).unwrap(),
            Array2::from_shape_vec((self.n, k), dist).unwrap(),
        )
    }

    /// reference src/ball_tree.rs:351-353
    pub fn num_points(&self) -> usize {
        self.n
    }

    /// A second handle onto the same device-resident tree with its own stream and workspaces (`pn_tree_session`):
    /// queries through `&self` from several threads are legal but serialise inside the library; give every thread
    /// its own session and they overlap on the GPU.  Nothing of the tree is copied.
    pub fn session(&self) -> Self {
        let mut h = std::ptr::null_mut();
        check(unsafe { ffi::pn_tree_session(self.handle.0, &mut h) });
        Self { handle: Handle(h), n: self.n, d: self.d, metric: Euclidean::default(), _p: PhantomData }
    }
}

/// Vantage-point tree (reference src/vantage_point_tree.rs).
pub struct VantagePointTree<'a, A, M = Euclidean> {
    handle: Handle,
    d: usize,
    #[allow(dead_code)]
    metric: M,
    _p: PhantomData<&'a A>,
}

impl<'a, A: Element> VantagePointTree<'a, A, Euclidean> {
    /// reference src/vantage_point_tree.rs:31-36
    pub fn euclidean<T: Into<CowArray<'a, A, Ix2>>>(points: T) -> Result<Self, ArrayError> {
        Self::new(points, Euclidean::default())
    }

    /// reference src/vantage_point_tree.rs:51-72
    pub fn new<T: Into<CowArray<'a, A, Ix2>>>(points: T, metric: Euclidean) -> Result<Self, ArrayError> {
        let points: CowArray<'a, A, Ix2> = points.into();
        let d = points.ncols();
        let mut h = std::ptr::null_mut();
        check_create(with_points(&points, |p, n, d, rs, cs| unsafe { A::vp_create(p, n, d, rs, cs, std::ptr::null(), &mut h) }))?;
        Ok(Self { handle: Handle(h), d, metric, _p: PhantomData })
    }

    /// reference src/vantage_point_tree.rs:88-98
    pub fn query_nearest<S: Data<Elem = A>>(&self, needle: &ArrayBase<S, Ix1>) -> (usize, A) {
        check_dim(needle.len(), self.d, "needle");
        let q = needle.to_owned();
        let (mut i, mut dist) = (0u64, A::zero());
        check(unsafe { A::vp_nearest(self.handle.0, q.as_ptr(), 1, self.d, &mut i, &mut dist) });
        (i as usize, dist)
    }

    pub fn query_nearest_batch(&self, queries: &ArrayView2<A>) -> (Array1<usize>, Array1<A>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        let nq = q.nrows();
        let mut idx = vec![0u64; nq];
        let mut dist = vec![A::zero(); nq];
        check(unsafe { A::vp_nearest(self.handle.0, q.as_ptr(), nq, self.d, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        (idx.into_iter().map(|i| i as usize).collect(), Array1::from_vec(dist))
    }

    /// Extension (the reference tree has `query_nearest` only): the `k` nearest neighbours, as `BallTree::query`
    /// returns them for the same points.
    pub fn query<S: Data<Elem = A>>(&self, point: &ArrayBase<S, Ix1>, k: usize) -> (Vec<usize>, Vec<A>) {
        check_dim(point.len(), self.d, "point");
        if k == 0 {
            return (Vec::new(), Vec::new());
        }
        let q = point.to_owned();
        let mut idx = vec![0u64; k];
        let mut dist = vec![A::zero(); k];
        check(unsafe { A::vp_query(self.handle.0, q.as_ptr(), 1, self.d, k, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        let m = idx.iter().take_while(|&&i| i != u64::MAX).count(); // rows are padded when k > n
        (idx[..m].iter().map(|&i| i as usize).collect(), dist[..m].to_vec())
    }

    /// Extension: all points with `distance < radius` (strict), indices ascending, as `BallTree::query_radius`.
    pub fn query_radius<S: Data<Elem = A>>(&self, point: &ArrayBase<S, Ix1>, distance: A) -> Vec<usize> {
        check_dim(point.len(), self.d, "point");
        let q = point.to_owned();
        let (mut po, mut pi) = (std::ptr::null_mut::<u64>(), std::ptr::null_mut::<u64>());
        check(unsafe { A::vp_radius(self.handle.0, q.as_ptr(), 1, self.d, distance, &mut po, &mut pi) });
        let total = unsafe { *po.add(1) } as usize;
        let out = (0..total).map(|i| unsafe { *pi.add(i) } as usize).collect();
        unsafe {
            ffi::pn_free(po as *mut std::ffi::c_void);
            ffi::pn_free(pi as *mut std::ffi::c_void);
        }
        out
    }
}

/// How a [`MultiGpuBallTree`] spreads over the devices.
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub enum ShardMode {
    /// the tree is replicated (built once, sent with ncclBroadcast), a batch of queries is split into slices
    Replicate,
    /// one depth-log2(n) subtree per device; per-shard lists are exchanged over NCCL and merged
    BySubtree,
}

/// Ball tree over several GPUs of one box, driven from this one process (`pn_multi_*`).  An addition to the reference
/// API: `query_batch` has the same result layout as [`BallTree::query_batch`].
pub struct MultiGpuBallTree {
    handle: *mut ffi::pn_multi,
    d: usize,
}
unsafe impl Send for MultiGpuBallTree {}

impl MultiGpuBallTree {
    pub fn euclidean(devices: &[i32], points: &ArrayView2<f32>, mode: ShardMode) -> Result<Self, ArrayError> {
        let p = points.as_standard_layout();
        let (n, d) = (p.nrows(), p.ncols());
        let mut h = std::ptr::null_mut();
        let m = if mode == ShardMode::Replicate { ffi::PN_SHARD_REPLICATE } else { ffi::PN_SHARD_BY_SUBTREE };
        check_create(unsafe {
            ffi::pn_multi_balltree_create_f32(devices.as_ptr(), devices.len() as i32, m, p.as_ptr(), n, d, d.max(1), std::ptr::null(), &mut h)
        })?;
        Ok(Self { handle: h, d })
    }

    pub fn query_batch(&mut self, queries: &ArrayView2<f32>, k: usize) -> (Array2<usize>, Array2<f32>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        let nq = q.nrows();
        let mut idx = vec![0u64; nq * k];
        let mut dist = vec![0f32; nq * k];
        check(unsafe { ffi::pn_multi_balltree_query_f32(self.handle, q.as_ptr(), nq, self.d, k, idx.as_mut_ptr(), dist.as_mut_ptr()) });
        (
            Array2::from_shape_vec((nq, k), idx.into_iter().map(|i| i as usize).collect()).unwrap(),
            Array2::from_shape_vec((nq, k), dist).unwrap(),
        )
    }

    /// Batched radius search over all devices: CSR `(offsets[nq + 1], indices)`, as [`BallTree::query_radius_batch`]
    /// returns it for a tree of all the points.
    pub fn query_radius_batch(&mut self, queries: &ArrayView2<f32>, distance: f32) -> (Vec<usize>, Vec<usize>) {
        check_dim(queries.ncols(), self.d, "query batch");
        let q = queries.as_standard_layout();
        let nq = q.nrows();
        let (mut po, mut pi) = (std::ptr::null_mut::<u64>(), std::ptr::null_mut::<u64>());
        check(unsafe { ffi::pn_multi_balltree_query_radius_f32(self.handle, q.as_ptr(), nq, self.d, distance, &mut po, &mut pi) });
        unsafe {
            let offsets: Vec<usize> = std::slice::from_raw_parts(po, nq + 1).iter().map(|&v| v as usize).collect();
            let total = *offsets.last().unwrap();
            let indices: Vec<usize> = std::slice::from_raw_parts(pi, total).iter().map(|&v| v as usize).collect();
            ffi::pn_free(po.cast());
            ffi::pn_free(pi.cast());
            (offsets, indices)
        }
    }
}

impl Drop for MultiGpuBallTree {
    fn drop(&mut self) {
        unsafe { ffi::pn_multi_destroy(self.handle) };
    }
}

#[cfg(test)]
mod test {
    // The reference's own doctests / unit tests, unchanged, run against the GPU crate.
    use ndarray::{array, aview1};

    use super::*;

    #[test]
    fn readme_example() {
        let points = array![[1., 1.], [1., 2.], [9., 9.]];
        let tree = BallTree::euclidean(points).expect("non-empty input");
        let (indices, _) = tree.query(&aview1(&[3., 3.]), 2);
        assert_eq!(indices, &[1, 0]);
        let (index, distance) = tree.query_nearest(&aview1(&[8., 8.]));
        assert_eq!(index, 2);
        assert!((2_f64.sqrt() - distance).abs() < 1e-8);
    }

    #[test]
    fn query_radius_doc() {
        let points = array![[1., 0.], [2., 0.], [9., 0.]];
        let tree = BallTree::euclidean(points).expect("non-empty input");
        assert_eq!(tree.query_radius(&aview1(&[3., 0.]), 1.5), &[1]);
    }

    #[test]
    fn vp_euclidian() {
        let points = array![[1.0, 2.0], [1.1, 2.2], [0.9, 1.9], [1.0, 2.1], [-2.0, 3.0], [-2.2, 3.1]];
        let vp = VantagePointTree::euclidean(points).expect("valid array");
        assert_eq!(vp.query_nearest(&aview1(&[0.95, 1.96])).0, 0);
    }
}
