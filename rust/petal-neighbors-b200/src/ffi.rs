//! Raw bindings of include/petal_b200.h (ABI version 1).
#![allow(non_camel_case_types)]
use std::os::raw::c_char;

pub const PN_OK: i32 = 0;
pub const PN_EMPTY: i32 = 1;
pub const PN_NOT_CONTIGUOUS: i32 = 2;

#[repr(C)]
pub struct pn_tree {
    _private: [u8; 0],
}

#[repr(C)]
#[derive(Default, Clone, Copy)]
pub struct pn_build_opts {
    pub struct_size: u32,
    pub device: i32,
    pub bucket_size: u32,
    pub algo: u32,
    pub host_threads: u32,
    pub flags: u32,
    pub shard_depth: u32,
    pub shard_index: u32,
    pub builder: u32, // pn_builder: 0 auto, 1 host, 2 device
    pub prune: u32,   // pn_prune: 0 auto, 1 on, 2 off
    pub partition: u32, // pn_partition: 0 auto, 1 reference, 2 two-means
    pub reserved: [u32; 5],
}

extern "C" {
    pub fn pn_last_error_message() -> *const c_char;
    pub fn pn_balltree_create_f32(p: *const f32, n: usize, d: usize, row_stride: usize, col_stride: usize,
                                  opts: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    pub fn pn_balltree_create_f64(p: *const f64, n: usize, d: usize, row_stride: usize, col_stride: usize,
                                  opts: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    pub fn pn_vptree_create_f32(p: *const f32, n: usize, d: usize, row_stride: usize, col_stride: usize,
                                opts: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    pub fn pn_vptree_create_f64(p: *const f64, n: usize, d: usize, row_stride: usize, col_stride: usize,
                                opts: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    pub fn pn_tree_destroy(t: *mut pn_tree) -> i32;
    pub fn pn_tree_session(t: *mut pn_tree, out: *mut *mut pn_tree) -> i32;
    pub fn pn_balltree_query_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize, k: usize,
                                 idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_balltree_query_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize, k: usize,
                                 idx: *mut u64, dist: *mut f64) -> i32;
    pub fn pn_balltree_query_nearest_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize,
                                         idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_balltree_query_nearest_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize,
                                         idx: *mut u64, dist: *mut f64) -> i32;
    pub fn pn_balltree_query_radius_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize, r: f32,
                                        offsets: *mut *mut u64, indices: *mut *mut u64) -> i32;
    pub fn pn_balltree_query_radius_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize, r: f64,
                                        offsets: *mut *mut u64, indices: *mut *mut u64) -> i32;
    pub fn pn_vptree_query_nearest_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize,
                                       idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_vptree_query_nearest_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize,
                                       idx: *mut u64, dist: *mut f64) -> i32;
    pub fn pn_vptree_query_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize, k: usize,
                               idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_vptree_query_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize, k: usize,
                               idx: *mut u64, dist: *mut f64) -> i32;
    pub fn pn_vptree_query_radius_f32(t: *mut pn_tree, q: *const f32, nq: usize, q_row_stride: usize, r: f32,
                                      offsets: *mut *mut u64, indices: *mut *mut u64) -> i32;
    pub fn pn_vptree_query_radius_f64(t: *mut pn_tree, q: *const f64, nq: usize, q_row_stride: usize, r: f64,
                                      offsets: *mut *mut u64, indices: *mut *mut u64) -> i32;
    pub fn pn_balltree_query_self_f32(t: *mut pn_tree, k: usize, idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_balltree_query_self_f64(t: *mut pn_tree, k: usize, idx: *mut u64, dist: *mut f64) -> i32;
    pub fn pn_free(p: *mut std::ffi::c_void);
    // one process, several GPUs (include/petal_b200.h: pn_multi_*)
    pub fn pn_multi_balltree_create_f32(devices: *const i32, n_dev: i32, shard_mode: u32, p: *const f32, n: usize, d: usize,
                                        row_stride: usize, opts: *const pn_build_opts, out: *mut *mut pn_multi) -> i32;
    pub fn pn_multi_balltree_query_f32(m: *mut pn_multi, q: *const f32, nq: usize, q_row_stride: usize, k: usize,
                                       idx: *mut u64, dist: *mut f32) -> i32;
    pub fn pn_multi_balltree_query_radius_f32(m: *mut pn_multi, q: *const f32, nq: usize, q_row_stride: usize, radius: f32,
                                              offsets: *mut *mut u64, indices: *mut *mut u64) -> i32;
    pub fn pn_multi_destroy(m: *mut pn_multi) -> i32;
    // merge of per-shard CSR radius results on one device (all pointers are device pointers)
    pub fn pn_merge_radius_dev(device: i32, offsets_lists_dev: *const u64, indices_lists_dev: *const u64, n_lists: usize, nq: usize,
                               out_offsets_dev: *mut u64, out_indices_dev: *mut u64, stream: *mut std::ffi::c_void, sync: i32) -> i32;
    // radius search from and into device memory on the tree's device (include/petal_b200.h: pn_tree_query_radius_dev)
    pub fn pn_tree_query_radius_dev(t: *mut pn_tree, queries_dev: *const std::ffi::c_void, nq: usize, q_row_stride: usize,
                                    radius: f64, offsets_dev: *mut u64, indices_dev: *mut u64, capacity: usize,
                                    stream: *mut std::ffi::c_void, sync: i32) -> i32;
}

#[repr(C)]
pub struct pn_multi {
    _private: [u8; 0],
}
pub const PN_SHARD_REPLICATE: u32 = 0;
pub const PN_SHARD_BY_SUBTREE: u32 = 1;

/// Element types the engine is instantiated for (the reference is generic over `A: Float`).
pub trait Element: Copy + num_traits::Float + 'static {
    unsafe fn ball_create(p: *const Self, n: usize, d: usize, rs: usize, cs: usize, o: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    unsafe fn vp_create(p: *const Self, n: usize, d: usize, rs: usize, cs: usize, o: *const pn_build_opts, out: *mut *mut pn_tree) -> i32;
    unsafe fn ball_query(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, k: usize, idx: *mut u64, dist: *mut Self) -> i32;
    unsafe fn ball_nearest(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, idx: *mut u64, dist: *mut Self) -> i32;
    unsafe fn ball_radius(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, r: Self, o: *mut *mut u64, i: *mut *mut u64) -> i32;
    unsafe fn vp_nearest(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, idx: *mut u64, dist: *mut Self) -> i32;
    unsafe fn ball_self(t: *mut pn_tree, k: usize, idx: *mut u64, dist: *mut Self) -> i32;
    unsafe fn vp_query(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, k: usize, idx: *mut u64, dist: *mut Self) -> i32;
    unsafe fn vp_radius(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, r: Self, o: *mut *mut u64, i: *mut *mut u64) -> i32;
}

macro_rules! impl_element {
    ($t:ty, $bc:ident, $vc:ident, $bq:ident, $bn:ident, $br:ident, $vn:ident, $bs:ident, $vq:ident, $vr:ident) => {
        impl Element for $t {
            unsafe fn ball_create(p: *const Self, n: usize, d: usize, rs: usize, cs: usize, o: *const pn_build_opts, out: *mut *mut pn_tree) -> i32 { $bc(p, n, d, rs, cs, o, out) }
            unsafe fn vp_create(p: *const Self, n: usize, d: usize, rs: usize, cs: usize, o: *const pn_build_opts, out: *mut *mut pn_tree) -> i32 { $vc(p, n, d, rs, cs, o, out) }
            unsafe fn ball_query(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, k: usize, idx: *mut u64, dist: *mut Self) -> i32 { $bq(t, q, nq, qs, k, idx, dist) }
            unsafe fn ball_nearest(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, idx: *mut u64, dist: *mut Self) -> i32 { $bn(t, q, nq, qs, idx, dist) }
            unsafe fn ball_radius(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, r: Self, o: *mut *mut u64, i: *mut *mut u64) -> i32 { $br(t, q, nq, qs, r, o, i) }
            unsafe fn vp_nearest(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, idx: *mut u64, dist: *mut Self) -> i32 { $vn(t, q, nq, qs, idx, dist) }
            unsafe fn ball_self(t: *mut pn_tree, k: usize, idx: *mut u64, dist: *mut Self) -> i32 { $bs(t, k, idx, dist) }
            unsafe fn vp_query(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, k: usize, idx: *mut u64, dist: *mut Self) -> i32 { $vq(t, q, nq, qs, k, idx, dist) }
            unsafe fn vp_radius(t: *mut pn_tree, q: *const Self, nq: usize, qs: usize, r: Self, o: *mut *mut u64, i: *mut *mut u64) -> i32 { $vr(t, q, nq, qs, r, o, i) }
        }
    };
}
impl_element!(f32, pn_balltree_create_f32, pn_vptree_create_f32, pn_balltree_query_f32, pn_balltree_query_nearest_f32, pn_balltree_query_radius_f32, pn_vptree_query_nearest_f32, pn_balltree_query_self_f32, pn_vptree_query_f32, pn_vptree_query_radius_f32);
impl_element!(f64, pn_balltree_create_f64, pn_vptree_create_f64, pn_balltree_query_f64, pn_balltree_query_nearest_f64, pn_balltree_query_radius_f64, pn_vptree_query_nearest_f64, pn_balltree_query_self_f64, pn_vptree_query_f64, pn_vptree_query_radius_f64);
